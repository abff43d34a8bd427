"""skani's --ci bootstrap interval of the ANI (DESIGN.md section 3): the shim's parser, the CPU reference
(tests/ani_ci_ref.py, on the oracle's accepted chains) against an independent statement of the definition (numpy
draws, replicates ranked by exact fractions and selected by sorting), and the device path against the CPU reference in
every finalize route, in every entry point and end to end through the shim."""
import itertools
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ani_ci_ref as REF  # noqa: E402
from test_ani_estimators import mag_queries, spread_pair  # noqa: E402

ACGT = np.frombuffer(b"ACGT", np.uint8)


def one_chain_pair(seed=5):
    """a 15 kb genome (one query chunk) and a copy with 1 % substitutions: one chain"""
    rng = np.random.default_rng(seed)
    ref = ACGT[rng.integers(0, 4, 15_000)]
    q = ref.copy()
    pos = np.nonzero(rng.random(len(q)) < 0.01)[0]
    q[pos] = ACGT[(np.searchsorted(ACGT, q[pos]) + rng.integers(1, 4, len(pos))) % 4]
    return [ref.tobytes()], [q.tobytes()]


# ---- the definition, restated independently ---------------------------------------------------------------------------
def _mix(z):
    """splitmix64 finalizer on uint64 arrays (numpy wraps mod 2^64)"""
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def expected_picks(chains):
    """(A, S) of the 5th- and 95th-percentile replicates: all draws at once in numpy, the replicates sorted by
    (Fraction(A_b, S_b), b)"""
    ch = sorted(chains, key=lambda c: (c.chunk, -c.score, c.q0, c.r0))
    a = np.array([c.n_anchors - 2 for c in ch], np.int64)
    s = np.array([c.n_seeds - 2 for c in ch], np.int64)
    n = len(ch)
    u = lambda v: np.array([v], np.uint64)  # noqa: E731 -- one-element arrays: scalar uint64 overflow would warn
    seed = _mix(_mix(_mix(u(n)) ^ u(int(a.sum()))) ^ u(int(s.sum())))
    b = np.arange(100, dtype=np.uint64)[:, None]
    i = np.arange(n, dtype=np.uint64)[None, :]
    z = _mix(seed ^ (b << np.uint64(40)) ^ i)
    # floor(z * n / 2^64) with n < 2^32: (hi * n + (lo * n >> 32)) >> 32, nothing overflows
    nn = np.uint64(n)
    j = ((z >> np.uint64(32)) * nn + (((z & np.uint64(0xFFFFFFFF)) * nn) >> np.uint64(32))) >> np.uint64(32)
    A, S = a[j.astype(np.int64)].sum(1), s[j.astype(np.int64)].sum(1)
    order = sorted(range(100), key=lambda k: (Fraction(int(A[k]), int(S[k])), k))
    return (int(A[order[5]]), int(S[order[5]])), (int(A[order[94]]), int(S[order[94]]))


def _check_ref_pair(O, x, y):
    """the reference's interval of (x, y) equals the restatement's, and (y, x) gets the same one; returns
    (ani, lo, hi, n_chains) as fractions, or None without an estimate"""
    r = O.pair(x, y)
    if r.ani < 0:
        assert REF.interval(x, y) is None
        return None
    _, chains = O.pair(x, y, want_chains=True, max_chains=r.n_chains + 16)
    assert len(chains) == r.n_chains
    want = expected_picks(chains)
    assert REF.picks(REF.replicates(chains)) == want
    lo, hi = REF.interval(x, y)
    assert (lo, hi) == tuple(min(1.0, REF.debias(float(min(Fraction(1), Fraction(A, S))) ** (1.0 / 15))) for A, S in want)
    assert REF.interval(y, x) == (lo, hi)
    return r.ani, lo, hi, r.n_chains


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_parser_accepts_ci():
    from skder_b200 import cli

    for argv in ("triangle -l L -E -o o", "dist --rl R --ql Q -o o", "search q.fa -d db -o o"):
        assert cli.parse_args(argv.split())[1]["ci"] is False
        sub, o = cli.parse_args((argv + " --ci").split())
        assert o["ci"] is True and o["estimator"] == "mean"
        for mode in ("median", "robust"):
            with pytest.raises(cli.UsageError):
                cli.parse_args((argv + " --ci --" + mode).split())
            with pytest.raises(cli.UsageError):
                cli.parse_args((argv + " --" + mode + " --ci").split())
    with pytest.raises(cli.UsageError):
        cli.parse_args("sketch -l L -o db --ci".split())
    assert cli.header(False) == cli.HEADER
    assert cli.header(True) == cli.HEADER[:-1] + "\tANI_5_percentile\tANI_95_percentile\n"


def test_cpu_reference_follows_the_definition(oracle, genomes7):
    from skder_b200 import synth

    O = oracle
    sk7 = [O.Sketch.from_file(f) for f in genomes7]
    for i, j in itertools.combinations(range(7), 2):
        _check_ref_pair(O, sk7[i], sk7[j])
    clade = [O.Sketch.from_contigs(c) for c in synth.one_clade(0, 4, 400_000, 77)]
    widths = []
    for i, j in itertools.combinations(range(4), 2):
        got = _check_ref_pair(O, clade[i], clade[j])
        widths.append(got[2] - got[1])
    a, b = spread_pair()
    ani, lo, hi, _ = _check_ref_pair(O, O.Sketch.from_contigs(a), O.Sketch.from_contigs(b))
    # the spread pair's chains differ in identity by up to 6 %: its interval brackets the ANI and is wider than any of
    # a clade's (about 1.1 pp against at most 0.4)
    assert lo < ani < hi
    assert hi - lo > 2 * max(widths)
    a, b = one_chain_pair()
    ani, lo, hi, n = _check_ref_pair(O, O.Sketch.from_contigs(a), O.Sketch.from_contigs(b))
    assert n == 1 and lo == hi == ani


def _run(script, argv, env=None):
    return subprocess.call([sys.executable, script] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **(env or {})))


def test_cpu_skani_takes_ci(oracle, genomes7, tmp_path):
    """the CPU `skani` the shim is compared with: with --ci its first seven columns are tests/oracle_skani.py's output
    byte for byte, and the two new ones are the reference's interval"""
    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in genomes7))
    plain, ci = tmp_path / "plain.tsv", tmp_path / "ci.tsv"
    argv = ["triangle", "-l", str(lst), "-E", "-t", "4"]
    assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"), argv + ["-o", str(plain)]) == 0
    assert _run(os.path.join(ROOT, "tests", "ani_ci_ref.py"), argv + ["--ci", "-o", str(ci)]) == 0
    p_rows = [ln.split("\t") for ln in plain.read_text().splitlines()]
    c_rows = [ln.split("\t") for ln in ci.read_text().splitlines()]
    assert len(c_rows) == len(p_rows) > 1
    assert c_rows[0] == p_rows[0] + ["ANI_5_percentile", "ANI_95_percentile"]
    assert [r[:7] for r in c_rows] == p_rows
    sk = {p: oracle.Sketch.from_file(p) for p in genomes7}
    for r in c_rows[1:]:
        assert r[7:] == ["%.2f" % (100 * v) for v in REF.interval(sk[r[0]], sk[r[1]])]


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _ci_of(edges, ci):
    return {(int(x["a"]), int(x["b"])): (float(lo), float(hi)) for x, (lo, hi) in zip(edges, ci)}


@pytest.mark.gpu
def test_rect_intervals_equal_reference_in_every_route(oracle, built_lib, genomes7):
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
            eng.set_ci(True)
            every = list(range(len(sk)))
            edges, _ = eng.rect(every if refs is None else refs, every if queries is None else queries, screen=0.0, min_af=0.0)
            ci = eng.last_edge_ci()
            assert ci.shape == (len(edges), 2) and len(edges) > 0, name
            for x, (lo, hi) in zip(edges, ci):
                want = REF.interval(sk[int(x["a"])], sk[int(x["b"])])
                assert abs(lo - 100 * want[0]) <= 1e-12 and abs(hi - 100 * want[1]) <= 1e-12, (name, x)
                assert ("%.2f" % lo, "%.2f" % hi) == ("%.2f" % (100 * want[0]), "%.2f" % (100 * want[1])), (name, x)
                if name == "one chain":
                    assert lo == hi == x["ani"]
            if name == "routes":
                # the warp kernel, the shared-memory CTA kernel (<= 4,096 candidates) and the global-scratch one
                det = eng.pairs_detail([0, 0, 0], [1, 2, 3])
                assert 1024 < det[0].n_chains <= 1500 and det[1].n_chains > 4096 and det[2].n_chains <= 1024


@pytest.fixture(scope="module")
def eng7(built_lib, genomes7):
    from skder_b200 import engine

    e = engine.Engine(0)
    packed = e.add_fasta(genomes7, threads=4)
    e.index()
    yield e, packed
    e.close()


@pytest.mark.gpu
def test_same_pair_same_interval_everywhere(eng7):
    """triangle, rect, search and a two-shard pairs_edges run give a pair the same interval, bit for bit"""
    from skder_b200 import engine

    e, packed = eng7
    e.set_ci(True)
    try:
        tri, _ = e.triangle(screen=80.0, min_af=15.0)
        want = _ci_of(tri, e.last_edge_ci())
        assert len(want) > 1
        rect, _ = e.rect(list(range(7)), list(range(7)), screen=80.0, min_af=15.0)
        for (a, b), iv in _ci_of(rect, e.last_edge_ci()).items():
            assert iv == want[min(a, b), max(a, b)]
        for k in (1, 4):
            edges, _ = e.search(packed[k], screen=80.0, min_af=15.0)
            got = _ci_of(edges, e.last_edge_ci())  # a = database genome, b = the query (a copy of genome k)
            assert {a for a, _ in got} - {k} == {a if b == k else b for a, b in want if k in (a, b)}
            for (a, _), iv in got.items():
                if a != k:
                    assert iv == want[min(a, k), max(a, k)]
    finally:
        e.set_ci(False)
    got = {}
    for first, count in [(0, 3), (3, 4)]:
        with engine.Engine(0) as e2:
            e2.set_ci(True)
            e2.add(packed)
            e2.index()
            e2.set_owned(first, count)
            e2.index()
            ptr, n, _ = e2.screen_triangle(80.0)
            e2.pairs_edges(ptr, n, owned_only=True, min_af=15.0, to_host=False)  # a result left on the device ...
            ci_dev = e2.last_edge_ci()
            assert len(ci_dev) == e2.device_edges()[1]
            edges, _ = e2.pairs_edges(ptr, n, owned_only=True, min_af=15.0)
            ci = e2.last_edge_ci()
            assert ci.tobytes() == ci_dev.tobytes()  # ... has the same intervals
            got.update(_ci_of(edges, ci))
    assert got == want


@pytest.mark.gpu
def test_ci_leaves_no_state_behind(eng7):
    from skder_b200 import engine
    from skder_b200._lib import SkbError

    e, packed = eng7
    runs = {}
    for on in (False, True, False):
        e.set_ci(on)
        l0 = e.launches
        edges, _ = e.triangle(screen=80.0, min_af=15.0)
        runs[on] = (e.launches - l0, edges.tobytes())
    e.set_ci(False)
    with pytest.raises(SkbError, match=r"\(-5\)"):  # SKB_ESTATE: the last call ran without --ci
        e.last_edge_ci()
    assert runs[True][1] == runs[False][1]  # the edges are the same with the interval on
    with engine.Engine(0) as fresh:
        fresh.add(packed)
        fresh.index()
        with pytest.raises(SkbError, match=r"\(-5\)"):  # no call yet
            fresh.last_edge_ci()
        l0 = fresh.launches
        want, _ = fresh.triangle(screen=80.0, min_af=15.0)
        assert (fresh.launches - l0, want.tobytes()) == runs[False]  # no launch added once it is off again
        # context state that survives clear()
        e.set_ci(True)
        e.triangle(screen=80.0, min_af=15.0)
        ci_e = e.last_edge_ci()
        e.set_ci(False)
        fresh.set_ci(True)
        fresh.clear()
        fresh.add(packed)
        fresh.index()
        fresh.triangle(screen=80.0, min_af=15.0)
        assert fresh.last_edge_ci().tobytes() == ci_e.tobytes()
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
            fresh.set_ci(False)
            fresh.triangle(screen=80.0, min_af=15.0)  # the median alone is fine
        finally:
            fresh.set_estimator("mean")


@pytest.mark.gpu
def test_shim_end_to_end_equals_cpu_skani(genomes7, built_lib, tmp_path):
    from skder_b200 import daemon

    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    cpu = os.path.join(ROOT, "tests", "ani_ci_ref.py")  # tests/oracle_skani.py, with the interval columns under --ci
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

    out = both(["triangle", "-l", str(lst), "--min-af", "15.0", "-E", "-t", "4", "--ci"])
    assert "--ci" in open(str(out) + ".skani_b200.log").read()
    assert len(out.read_text().splitlines()[1].split("\t")) == 9
    both(["dist", "--rl", str(rl), "--ql", str(ql), "--ci"])
    db = tmp_path / "db"
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(db), "-t", "4"]) == 0
    q = genomes7[2]
    both(["search", q, "-d", str(db), "-t", "2", "--ci"], {"SKB_NO_DAEMON": "1"})
    try:
        for extra in (["--ci"], [], ["--ci"], []):  # one resident server alternates
            both(["search", q, "-d", str(db), "-t", "2"] + extra, {"SKB_DAEMON_IDLE": "120"})
        assert daemon.request(str(db), 0, {"op": "ping"}, timeout=5.0)["n"] == 7
    finally:
        daemon.stop_for(str(db))
    bad = tmp_path / "bad.tsv"
    for argv in (["triangle", "-l", str(lst), "-E", "--ci", "--median"], ["dist", "--rl", str(rl), "--ql", str(ql), "--robust", "--ci"],
                 ["search", q, "-d", str(db), "--ci", "--median"]):
        assert _run(shim, argv + ["-o", str(bad)]) != 0 and not bad.exists()
    bad_db = tmp_path / "bad_db"
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(bad_db), "--ci"]) != 0 and not bad_db.exists()
