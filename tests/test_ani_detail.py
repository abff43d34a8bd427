"""skani's --detailed columns (DESIGN.md section 3): the shim's parser and header, the CPU reference
(tests/ani_detail_ref.py, on the oracle's accepted chains) against an independent restatement (numpy weighted averages,
sorts and cumulative sums), and the device path against the CPU reference in every finalize route, in every entry point
and end to end through the shim."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ani_ci_ref as CI  # noqa: E402
import ani_detail_ref as REF  # noqa: E402
from test_ani_ci import one_chain_pair  # noqa: E402
from test_ani_estimators import mag_queries, spread_pair  # noqa: E402

COLUMNS = ("Num_ref_contigs\tNum_query_contigs\tANI_5_percentile\tANI_95_percentile\tStandard_deviation\tRef_90_ctg_len\t"
           "Ref_50_ctg_len\tRef_10_ctg_len\tQuery_90_ctg_len\tQuery_50_ctg_len\tQuery_10_ctg_len\tAvg_chain_len\t"
           "Total_bases_covered")


# ---- the definition, restated independently ---------------------------------------------------------------------------
def expected_sd(chains):
    """numpy's weighted averages over the chains' own ANI (fraction)"""
    a = np.array([c.n_anchors - 2 for c in chains], np.float64)
    s = np.array([c.n_seeds - 2 for c in chains], np.float64)
    d = np.array([min(1.0, CI.debias(r ** (1.0 / 15))) for r in np.minimum(1.0, a / s)])
    mu = np.average(d, weights=s)
    return float(np.sqrt(np.average((d - mu) ** 2, weights=s)))


def expected_nx(lens):
    """(N90, N50, N10) by numpy sort and cumsum"""
    v = np.sort(np.asarray(lens, np.int64))[::-1]
    cs = np.cumsum(v)
    return tuple(int(v[np.argmax(100 * cs >= x * cs[-1])]) if len(v) else 0 for x in (90, 50, 10))


def _check_ref_pair(O, x, y):
    """the reference's detail of (x, y) against the restatement; returns (ani, detail) or None without an estimate"""
    r = O.pair(x, y)
    d = REF.detail(x, y)
    if r.ani < 0:
        assert d is None
        return None
    _, chains = O.pair(x, y, want_chains=True, max_chains=r.n_chains + 16)
    assert len(chains) == r.n_chains == d["n_chains"]
    assert abs(d["sd"] - expected_sd(chains)) <= 1e-12
    assert (d["lo"], d["hi"]) == CI.interval(x, y)
    for cov, af, g in ((d["covered_a"], r.af_a, x), (d["covered_b"], r.af_b, y)):
        if af < 1.0:  # the AF is this numerator over the genome's kept bases (capped at 100 %)
            assert abs(100.0 * cov / g.total_len - 100.0 * af) <= 1e-9
    for g in (x, y):
        assert REF.nx(g) == expected_nx(g.contig_lens())
        assert g.n_contigs == len(g.contig_lens())
    return r.ani, d


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_parser_accepts_detailed():
    from skder_b200 import cli

    for argv in ("triangle -l L -E -o o", "dist --rl R --ql Q -o o", "search q.fa -d db -o o"):
        assert cli.parse_args(argv.split())[1]["detailed"] is False
        for extra in (" --detailed", " --detailed --ci", " --ci --detailed"):
            sub, o = cli.parse_args((argv + extra).split())
            assert o["detailed"] is True and o["estimator"] == "mean" and o["ci"] == ("--ci" in extra)
        for mode in ("median", "robust"):
            with pytest.raises(cli.UsageError):
                cli.parse_args((argv + " --detailed --" + mode).split())
            with pytest.raises(cli.UsageError):
                cli.parse_args((argv + " --" + mode + " --detailed").split())
    with pytest.raises(cli.UsageError):
        cli.parse_args("sketch -l L -o db --detailed".split())
    want = cli.HEADER[:-1] + "\t" + COLUMNS + "\n"
    assert cli.header(False, True) == cli.header(True, True) == want
    assert len(want.split("\t")) == 20
    assert cli.header(False) == cli.HEADER
    assert cli.header(True) == cli.HEADER[:-1] + "\tANI_5_percentile\tANI_95_percentile\n"


def test_rows_carry_the_detail_through_the_sort():
    from skder_b200 import cli
    from skder_b200.engine import DETAIL_DTYPE, EDGE_DTYPE

    edges = np.array([(0, 2, 97.0, 80.0, 81.0), (1, 2, 99.0, 90.0, 91.0)], EDGE_DTYPE)
    det = np.zeros(2, DETAIL_DTYPE)
    det[["ani_lo", "ani_hi", "sd", "covered_a", "covered_b", "n_chains"]] = [(96.5, 97.5, 1.25, 10, 1001, 2),
                                                                            (98.5, 99.5, 0.5, 20, 3000, 3)]
    cnt = np.array([3, 4, 5], np.int32)
    nx = np.array([[1, 2, 3], [4, 5, 6], [7, 8, 9]], np.int64)
    detail = cli.edge_details(edges, det, cnt, nx)
    assert detail == [(3, 5, 96.5, 97.5, 1.25, 1, 2, 3, 7, 8, 9, 500, 1001),
                      (4, 5, 98.5, 99.5, 0.5, 4, 5, 6, 7, 8, 9, 1000, 3000)]
    rows = cli.rect_rows(["/r1", "/r2", "/q"], ["n1", "n2", "nq"], edges, None, detail)  # ANI descending: r2 first
    assert rows == ["/r2\t/q\t99.00\t90.00\t91.00\tn2\tnq\t4\t5\t98.50\t99.50\t0.50\t4\t5\t6\t7\t8\t9\t1000\t3000\n",
                    "/r1\t/q\t97.00\t80.00\t81.00\tn1\tnq\t3\t5\t96.50\t97.50\t1.25\t1\t2\t3\t7\t8\t9\t500\t1001\n"]
    assert cli.triangle_rows(["/a", "/b", "/c"], ["na", "nb", "nc"], edges, np.array([[1.0, 2.0], [3.0, 4.0]]),
                             detail)[0].endswith("\t1\t2\t3\t7\t8\t9\t500\t1001\n")  # the detail replaces --ci's columns


def test_cpu_reference_follows_the_definition(oracle, genomes7):
    from skder_b200 import synth

    O = oracle
    sk7 = [O.Sketch.from_file(f) for f in genomes7]
    for i, j in itertools.combinations(range(7), 2):
        _check_ref_pair(O, sk7[i], sk7[j])
    clade = [O.Sketch.from_contigs(c) for c in synth.one_clade(0, 4, 400_000, 77)]
    sds = [_check_ref_pair(O, clade[i], clade[j])[1]["sd"] for i, j in itertools.combinations(range(4), 2)]
    a, b = spread_pair()
    ani, d = _check_ref_pair(O, O.Sketch.from_contigs(a), O.Sketch.from_contigs(b))
    # the spread pair's chains differ in identity by up to 6 %: a spread well above a clade's
    assert d["sd"] > 0.015 and d["sd"] > 1.5 * max(sds)
    a, b = one_chain_pair()
    ani, d = _check_ref_pair(O, O.Sketch.from_contigs(a), O.Sketch.from_contigs(b))
    assert d["n_chains"] == 1 and d["sd"] == 0.0 and d["lo"] == d["hi"] == ani


def _run(script, argv, env=None):
    return subprocess.call([sys.executable, script] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **(env or {})))


def test_cpu_skani_takes_detailed(oracle, genomes7, tmp_path):
    """the CPU `skani` the shim is compared with: with --detailed its first seven columns are tests/oracle_skani.py's
    output byte for byte, its interval columns are tests/ani_ci_ref.py --ci's, and the rest is the reference's"""
    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in genomes7))
    plain, ci, det, det_ci = (tmp_path / n for n in ("plain.tsv", "ci.tsv", "det.tsv", "det_ci.tsv"))
    argv = ["triangle", "-l", str(lst), "-E", "-t", "4"]
    assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"), argv + ["-o", str(plain)]) == 0
    assert _run(os.path.join(ROOT, "tests", "ani_ci_ref.py"), argv + ["--ci", "-o", str(ci)]) == 0
    assert _run(os.path.join(ROOT, "tests", "ani_detail_ref.py"), argv + ["--detailed", "-o", str(det)]) == 0
    assert _run(os.path.join(ROOT, "tests", "ani_detail_ref.py"), argv + ["--detailed", "--ci", "-o", str(det_ci)]) == 0
    assert det.read_text() == det_ci.read_text()  # 20 columns, not 22
    p_rows = [ln.split("\t") for ln in plain.read_text().splitlines()]
    c_rows = [ln.split("\t") for ln in ci.read_text().splitlines()]
    d_rows = [ln.split("\t") for ln in det.read_text().splitlines()]
    assert len(d_rows) == len(p_rows) > 1
    assert d_rows[0] == p_rows[0] + COLUMNS.split("\t")
    assert [r[:7] for r in d_rows] == p_rows
    assert [r[9:11] for r in d_rows[1:]] == [r[7:9] for r in c_rows[1:]]
    sk = {p: oracle.Sketch.from_file(p) for p in genomes7}
    for r in d_rows[1:]:
        x, y = sk[r[0]], sk[r[1]]
        d = REF.detail(x, y)
        want = [x.n_contigs, y.n_contigs, None, None, "%.2f" % (100 * d["sd"]), *REF.nx(x), *REF.nx(y),
                d["covered_b"] // d["n_chains"], d["covered_b"]]
        assert [str(w) for w in want if w is not None] == r[7:9] + r[11:]


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _det_of(edges, det):
    """{(a, b): (lo, hi, sd, n_chains, {a: covered_a, b: covered_b})}"""
    return {(int(x["a"]), int(x["b"])): (float(d["ani_lo"]), float(d["ani_hi"]), float(d["sd"]), int(d["n_chains"]),
                                         {int(x["a"]): int(d["covered_a"]), int(x["b"]): int(d["covered_b"])})
            for x, d in zip(edges, det)}


@pytest.mark.gpu
def test_rect_detail_equals_reference_in_every_route(oracle, built_lib, genomes7):
    from skder_b200 import engine, synth

    O = oracle
    sets = [("genomes7", None, None, None)]
    sets.append(("clades", [c for _, _, c in synth.config_genomes("tiny")], None, None))
    a, b = spread_pair()
    sets.append(("spread", [a, b], None, None))
    c1, c2 = one_chain_pair()
    sets.append(("one chain", [c1, c2], None, None))
    sets.append(("routes", mag_queries(), [0], [1, 2, 3]))
    for name, contigs, refs, queries in sets:
        with engine.Engine(0) as eng:
            if contigs is None:
                eng.add_fasta(genomes7, threads=4)
                sk = [O.Sketch.from_file(p) for p in genomes7]
            else:
                eng.add([engine.pack_contigs(c) for c in contigs])
                sk = [O.Sketch.from_contigs(c) for c in contigs]
            eng.index()
            eng.set_detailed(True)
            every = list(range(len(sk)))
            edges, _ = eng.rect(every if refs is None else refs, every if queries is None else queries, screen=0.0, min_af=0.0)
            det = eng.last_edge_detail()
            assert det.shape == (len(edges),) and len(edges) > 0, name
            for x, d in zip(edges, det):
                want = REF.detail(sk[int(x["a"])], sk[int(x["b"])])
                for k in ("lo", "hi", "sd"):
                    got = d["ani_" + k] if k != "sd" else d["sd"]
                    assert abs(got - 100 * want[k]) <= 1e-12, (name, k, x)
                    assert "%.2f" % got == "%.2f" % (100 * want[k]), (name, k, x)
                assert (d["covered_a"], d["covered_b"], d["n_chains"]) == (want["covered_a"], want["covered_b"],
                                                                           want["n_chains"]), (name, x)
                if name == "one chain":
                    assert d["ani_lo"] == d["ani_hi"] == x["ani"] and d["sd"] == 0.0
            cnt, nx = eng.contig_stats(0, len(sk))
            assert cnt.tolist() == [s.n_contigs for s in sk], name
            assert [tuple(v) for v in nx.tolist()] == [REF.nx(s) for s in sk], name
            if name == "routes":
                # the warp kernel, the shared-memory CTA kernel (<= 4,096 candidates) and the global-scratch one
                pd = eng.pairs_detail([0, 0, 0], [1, 2, 3])
                assert 1024 < pd[0].n_chains <= 1500 and pd[1].n_chains > 4096 and pd[2].n_chains <= 1024
            if name == "spread":
                assert det["sd"].min() > 0.5  # percent


@pytest.fixture(scope="module")
def eng7(built_lib, genomes7):
    from skder_b200 import engine

    e = engine.Engine(0)
    packed = e.add_fasta(genomes7, threads=4)
    e.index()
    yield e, packed
    e.close()


def _same(got, want, flip):
    """a pair's detail equals another call's; flip maps got's genome ids to want's"""
    assert got[:4] == want[:4]
    assert {flip.get(g, g): v for g, v in got[4].items()} == want[4]


@pytest.mark.gpu
def test_same_pair_same_detail_everywhere(eng7):
    """triangle, rect, search and a two-shard pairs_edges run give a pair the same detail, bit for bit"""
    from skder_b200 import engine

    e, packed = eng7
    e.set_detailed(True)
    try:
        tri, _ = e.triangle(screen=80.0, min_af=15.0)
        want = _det_of(tri, e.last_edge_detail())
        assert len(want) > 1
        rect, _ = e.rect(list(range(7)), list(range(7)), screen=80.0, min_af=15.0)
        for (a, b), dt in _det_of(rect, e.last_edge_detail()).items():
            _same(dt, want[min(a, b), max(a, b)], {})
        for k in (1, 4):
            edges, _ = e.search(packed[k], screen=80.0, min_af=15.0)
            got = _det_of(edges, e.last_edge_detail())  # a = database genome, b = 7, the query (a copy of genome k)
            assert {a for a, _ in got} - {k} == {a if b == k else b for a, b in want if k in (a, b)}
            for (a, q), dt in got.items():
                if a != k:
                    _same(dt, want[min(a, k), max(a, k)], {q: k})
            cnt, nx = e.last_query_contig_stats
            want_cnt, want_nx = e.contig_stats(k, 1)
            assert cnt.tolist() == want_cnt.tolist() and nx.tolist() == want_nx.tolist()
    finally:
        e.set_detailed(False)
    got = {}
    for first, count in [(0, 3), (3, 4)]:
        with engine.Engine(0) as e2:
            e2.set_detailed(True)
            e2.add(packed)
            e2.index()
            e2.set_owned(first, count)
            e2.index()
            ptr, n, _ = e2.screen_triangle(80.0)
            e2.pairs_edges(ptr, n, owned_only=True, min_af=15.0, to_host=False)  # a result left on the device ...
            det_dev = e2.last_edge_detail()
            assert len(det_dev) == e2.device_edges()[1]
            edges, _ = e2.pairs_edges(ptr, n, owned_only=True, min_af=15.0)
            det = e2.last_edge_detail()
            assert det.tobytes() == det_dev.tobytes()  # ... has the same details
            got.update(_det_of(edges, det))
    assert got == want


@pytest.mark.gpu
def test_detailed_leaves_no_state_behind(eng7):
    from skder_b200 import engine
    from skder_b200._lib import SkbError

    e, packed = eng7
    runs = {}
    for on in (False, True, False):
        e.set_detailed(on)
        l0 = e.launches
        edges, _ = e.triangle(screen=80.0, min_af=15.0)
        runs[on] = (e.launches - l0, edges.tobytes())
    e.set_detailed(False)
    with pytest.raises(SkbError, match=r"\(-5\)"):  # SKB_ESTATE: the last call ran without --detailed
        e.last_edge_detail()
    assert runs[True][1] == runs[False][1]  # the edges are the same with it on
    assert runs[True][0] > runs[False][0]
    with engine.Engine(0) as fresh:
        fresh.add(packed)
        fresh.index()
        with pytest.raises(SkbError, match=r"\(-5\)"):  # no call yet
            fresh.last_edge_detail()
        l0 = fresh.launches
        want, _ = fresh.triangle(screen=80.0, min_af=15.0)
        assert (fresh.launches - l0, want.tobytes()) == runs[False]  # no launch added once it is off again
        # context state that survives clear()
        e.set_detailed(True)
        e.triangle(screen=80.0, min_af=15.0)
        det_e = e.last_edge_detail()
        with pytest.raises(SkbError, match=r"\(-5\)"):  # last_edge_ci keeps its meaning: --ci only
            e.last_edge_ci()
        # with --ci as well: last_edge_ci gives the detail's interval, bit for bit, and the detail does not change
        e.set_ci(True)
        try:
            e.triangle(screen=80.0, min_af=15.0)
            ci, det_ci = e.last_edge_ci(), e.last_edge_detail()
        finally:
            e.set_ci(False)
            e.set_detailed(False)
        assert det_ci.tobytes() == det_e.tobytes()
        assert ci.tobytes() == np.stack([det_e["ani_lo"], det_e["ani_hi"]], 1).tobytes()
        fresh.set_detailed(True)
        fresh.clear()
        fresh.add(packed)
        fresh.index()
        fresh.triangle(screen=80.0, min_af=15.0)
        assert fresh.last_edge_detail().tobytes() == det_e.tobytes()
        # defined for the mean only: SKB_EINVAL from every entry point, nothing computed
        fresh.set_estimator("median")
        try:
            with pytest.raises(SkbError, match=r"\(-1\)"):
                fresh.triangle(screen=80.0, min_af=15.0)
            with pytest.raises(SkbError, match=r"\(-1\)"):
                fresh.rect([0, 1], [2, 3], screen=80.0, min_af=15.0)
            ptr, n, _ = fresh.screen_triangle(80.0)
            with pytest.raises(SkbError, match=r"\(-1\)"):
                fresh.pairs_edges(ptr, n, owned_only=False, min_af=15.0)
            fresh.set_detailed(False)
            fresh.triangle(screen=80.0, min_af=15.0)  # the median alone is fine
        finally:
            fresh.set_estimator("mean")


@pytest.mark.gpu
def test_shim_end_to_end_equals_cpu_skani(genomes7, built_lib, tmp_path):
    from skder_b200 import daemon

    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    cpu = os.path.join(ROOT, "tests", "ani_detail_ref.py")  # the CPU skani, with --detailed's and --ci's columns
    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in genomes7))
    rl, ql = tmp_path / "r.txt", tmp_path / "q.txt"
    rl.write_text("".join(p + "\n" for p in genomes7[:4]))
    ql.write_text("".join(p + "\n" for p in genomes7[4:]))

    def both(argv, env=None):
        out, ref = tmp_path / "gpu.tsv", tmp_path / "cpu.tsv"
        for f in (out, ref):
            if f.exists():
                f.unlink()
        assert _run(shim, argv + ["-o", str(out)], env) == 0
        assert _run(cpu, argv + ["-o", str(ref)]) == 0
        assert out.read_text() == ref.read_text(), argv
        return out

    out = both(["triangle", "-l", str(lst), "--min-af", "15.0", "-E", "-t", "4", "--detailed"])
    log = open(str(out) + ".skani_b200.log").read()
    assert "--detailed" in log and "unpinned" in log
    assert len(out.read_text().splitlines()[1].split("\t")) == 20
    both(["triangle", "-l", str(lst), "--min-af", "15.0", "-E", "-t", "4", "--detailed", "--ci"])
    both(["dist", "--rl", str(rl), "--ql", str(ql), "--detailed"])
    db = tmp_path / "db"
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(db), "-t", "4"]) == 0
    q = genomes7[2]
    both(["search", q, "-d", str(db), "-t", "2", "--detailed"], {"SKB_NO_DAEMON": "1"})
    try:
        for extra in (["--detailed"], ["--ci"], [], ["--detailed"], ["--detailed", "--ci"], []):  # one resident server
            both(["search", q, "-d", str(db), "-t", "2"] + extra, {"SKB_DAEMON_IDLE": "120"})
        assert daemon.request(str(db), 0, {"op": "ping"}, timeout=5.0)["n"] == 7
    finally:
        daemon.stop_for(str(db))
    bad = tmp_path / "bad.tsv"
    for argv in (["triangle", "-l", str(lst), "-E", "--detailed", "--median"],
                 ["dist", "--rl", str(rl), "--ql", str(ql), "--robust", "--detailed"],
                 ["search", q, "-d", str(db), "--detailed", "--median"]):
        assert _run(shim, argv + ["-o", str(bad)]) != 0 and not bad.exists()
    bad_db = tmp_path / "bad_db"
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(bad_db), "--detailed"]) != 0 and not bad_db.exists()
