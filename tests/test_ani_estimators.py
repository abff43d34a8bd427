"""skani's --median and --robust ANI estimators (DESIGN.md section 3): the shim's parser, the CPU reference
(tests/ani_estimators_ref.py, on the oracle's accepted chains) against an independent statement of the definition in
exact fractions, and the device path against the CPU reference in every finalize route."""
import itertools
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ani_estimators_ref as REF  # noqa: E402

MODES = ("median", "robust")
ACGT = np.frombuffer(b"ACGT", np.uint8)


# ---- inputs -----------------------------------------------------------------------------------------------------------
def _mutate(seq, rate, rng):
    """substitutions at `rate` per base (a uint8 ACGT array in, bytes out)"""
    s = seq.copy()
    pos = np.nonzero(rng.random(len(s)) < rate)[0]
    s[pos] = ACGT[(np.searchsorted(ACGT, s[pos]) + rng.integers(1, 4, len(pos))) % 4]
    return s.tobytes()


def spread_pair(seed=3):
    """A genome and a copy whose 20 kb regions diverge at 0.2 .. 6 %: its chains have clearly spread identities."""
    rng = np.random.default_rng(seed)
    ref = ACGT[rng.integers(0, 4, 600_000)]
    rates = np.repeat(np.linspace(0.002, 0.06, 30), 20_000)
    rng.shuffle(rates.reshape(30, 20_000))
    q = ref.copy()
    pos = np.nonzero(rng.random(len(q)) < rates)[0]
    q[pos] = ACGT[(np.searchsorted(ACGT, q[pos]) + rng.integers(1, 4, len(pos))) % 4]
    return [ref.tobytes()], [q.tobytes()]


def mag_queries(seed=9):
    """An unfragmented source and two MAG-like copies with a divergence drawn per contig (0.2 .. 4 %): 1,500 contigs of
    3 kb (one chain each: more candidates than the warp kernel keeps, fewer than the shared-memory CTA kernel's 4,096)
    and 6,000 contigs of 1.5 kb (beyond 4,096: the global-scratch CTA kernel); plus a plain 300 kb relative."""
    rng = np.random.default_rng(seed)
    src = ACGT[rng.integers(0, 4, 9_000_000)]

    def frag(n, ln):
        return [_mutate(src[k * ln:(k + 1) * ln], rng.uniform(0.002, 0.04), rng) for k in range(n)]

    return [[src.tobytes()], frag(1500, 3000), frag(6000, 1500), [_mutate(src[:300_000], 0.01, rng)]]


# ---- the definition, restated independently with exact fractions -----------------------------------------------------
def expected_raw(chains, mode):
    """ANI_raw of `mode` from the accepted chains (oracle.pair(..., want_chains=True)), per DESIGN.md section 3."""
    ch = [(Fraction(c.n_anchors - 2, c.n_seeds - 2), c.chunk, -c.score, c.q0, c.r0, c.n_anchors - 2, c.n_seeds - 2)
          for c in chains]
    A, S = sum(c[5] for c in ch), sum(c[6] for c in ch)
    if mode == "mean":
        a, s = A, S
    else:
        ch.sort(key=lambda c: c[:5])
        W, C, a, s = S, 0, 0, 0
        for c in ch:
            C += c[6]
            if mode == "median" and 2 * C >= W:
                a, s = c[5], c[6]
                break
            if mode == "robust" and 10 * C > W and 10 * (C - c[6]) < 9 * W:
                a, s = a + c[5], s + c[6]
    return min(1.0, a / s) ** (1.0 / 15)


INT_FIELDS = ("n_chains", "swapped", "n_anchors_total", "n_seeds_total", "span_q", "span_r")


def _check_ref_pair(O, x, y):
    mean = O.pair(x, y)
    if mean.ani < 0:
        for mode in MODES:
            assert REF.pair(x, y, mode=mode).ani < 0
        return None
    _, chains = O.pair(x, y, want_chains=True, max_chains=mean.n_chains + 16)
    assert len(chains) == mean.n_chains
    assert abs(mean.ani_raw - expected_raw(chains, "mean")) <= 1e-12
    assert abs(REF.pair(x, y, mode="mean").ani_raw - mean.ani_raw) == 0
    got = {}
    for mode in MODES:
        r = REF.pair(x, y, mode=mode)
        assert abs(r.ani_raw - expected_raw(chains, mode)) <= 1e-12, mode
        assert r.ani == min(1.0, REF.debias(r.ani_raw))
        assert [getattr(r, f) for f in INT_FIELDS] == [getattr(mean, f) for f in INT_FIELDS]
        assert (r.af_a, r.af_b) == (mean.af_a, mean.af_b)
        got[mode] = r.ani_raw
    return mean.ani_raw, got


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_parser_accepts_median_and_robust():
    from skder_b200 import cli

    for argv in ("triangle -l L -E -o o", "dist --rl R --ql Q -o o", "search q.fa -d db -o o"):
        assert cli.parse_args(argv.split())[1]["estimator"] == "mean"
        for mode in MODES:
            sub, o = cli.parse_args((argv + " --" + mode).split())
            assert o["estimator"] == mode
        with pytest.raises(cli.UsageError):
            cli.parse_args((argv + " --median --robust").split())
    assert cli.parse_args("sketch -l L -o db".split())[1]["estimator"] == "mean"
    for mode in MODES:
        with pytest.raises(cli.UsageError):
            cli.parse_args(("sketch -l L -o db --" + mode).split())


def test_cpu_reference_follows_the_definition(oracle, genomes7):
    from skder_b200 import synth

    O = oracle
    sk7 = [O.Sketch.from_file(f) for f in genomes7]
    for i, j in itertools.combinations(range(7), 2):
        _check_ref_pair(O, sk7[i], sk7[j])
    clade = [O.Sketch.from_contigs(c) for c in synth.one_clade(0, 4, 400_000, 77)]
    for i, j in itertools.combinations(range(4), 2):
        _check_ref_pair(O, clade[i], clade[j])
    a, b = spread_pair()
    mean, got = _check_ref_pair(O, O.Sketch.from_contigs(a), O.Sketch.from_contigs(b))
    # the chains really are spread: trimming and the median select something the pooled mean does not
    assert got["robust"] > mean + 1e-4 and abs(got["median"] - mean) > 1e-4


def test_cpu_skani_takes_the_estimator(oracle, genomes7, tmp_path):
    """the CPU `skani` the shim is compared with: without a flag it is tests/oracle_skani.py byte for byte; with one,
    every row carries that estimator's ANI and the same AF"""
    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in genomes7))
    outs = {}
    for script, mode in (("oracle_skani.py", "mean"), ("ani_estimators_ref.py", "mean"), ("ani_estimators_ref.py", "robust")):
        out = tmp_path / ("%s.%s.tsv" % (script, mode))
        flag = [] if mode == "mean" else ["--" + mode]
        assert _run(os.path.join(ROOT, "tests", script), ["triangle", "-l", str(lst), "-E", "-o", str(out)] + flag) == 0
        outs[script, mode] = [ln.split("\t") for ln in out.read_text().splitlines()]
    assert outs["oracle_skani.py", "mean"] == outs["ani_estimators_ref.py", "mean"]
    rob, mean = outs["ani_estimators_ref.py", "robust"], outs["ani_estimators_ref.py", "mean"]
    assert [r[:2] + r[3:] for r in rob] == [r[:2] + r[3:] for r in mean] and len(rob) > 1
    sk = {p: oracle.Sketch.from_file(p) for p in genomes7}
    for r in rob[1:]:
        assert r[2] == "%.2f" % (REF.pair(sk[r[0]], sk[r[1]], mode="robust").ani * 100)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _detail_matches(d, r):
    assert (d.swapped, d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r) == (
        r.swapped, r.n_chains, r.n_anchors_total, r.n_seeds_total, r.span_q, r.span_r)
    assert (d.ani < 0) == (r.ani < 0)
    if r.ani >= 0:
        assert abs(d.ani_raw - r.ani_raw) <= 1e-12 and abs(d.ani - r.ani) <= 1e-12
        assert abs(d.af_a - r.af_a) < 1e-15 and abs(d.af_b - r.af_b) < 1e-15


@pytest.fixture(scope="module")
def eng7(built_lib, genomes7):
    from skder_b200 import engine

    e = engine.Engine(0)
    packed = e.add_fasta(genomes7, threads=4)
    e.index()
    yield e, packed
    e.set_estimator("mean")
    e.close()


@pytest.mark.gpu
def test_pairs_detail_equal_oracle_in_every_route(eng7, oracle, built_lib):
    from skder_b200 import engine, synth

    O = oracle
    e, _ = eng7
    sets = [("genomes7", None, list(itertools.combinations(range(7), 2)) + [(3, 1), (6, 0)])]
    sets.append(("clades", [c for _, _, c in synth.config_genomes("tiny")], None))
    a, b = spread_pair()
    sets.append(("spread", [a, b], [(0, 1)]))
    sets.append(("routes", mag_queries(), [(0, 1), (0, 2), (0, 3)]))
    for name, contigs, pairs in sets:
        if contigs is None:
            eng, sk = e, [O.Sketch.from_file(p.path) for p in eng7[1]]
        else:
            eng = engine.Engine(0)
            eng.add([engine.pack_contigs(c) for c in contigs])
            eng.index()
            sk = [O.Sketch.from_contigs(c) for c in contigs]
        if pairs is None:
            pairs = list(itertools.combinations(range(len(sk)), 2))
        try:
            for mode in ("mean",) + MODES:
                eng.set_estimator(mode)
                det = eng.pairs_detail([p[0] for p in pairs], [p[1] for p in pairs])
                for (i, j), d in zip(pairs, det):
                    _detail_matches(d, REF.pair(sk[i], sk[j], mode=mode))
                if name == "routes":
                    # accepted chains bound the candidates from below; one chain per contig bounds them from above
                    assert 1024 < det[0].n_chains <= 1500 and det[1].n_chains > 4096 and det[2].n_chains <= 1024
        finally:
            eng.set_estimator("mean")
            if eng is not e:
                eng.close()


def _cols(edges):
    return [edges[k].tolist() for k in ("a", "b", "af_a", "af_b")]


def _fmt(edges):
    return {(int(x["a"]), int(x["b"])): ("%.2f" % x["ani"], "%.2f" % x["af_a"], "%.2f" % x["af_b"]) for x in edges}


@pytest.mark.gpu
def test_triangle_and_rect_equal_cpu_reference(eng7, oracle):
    from oracle import skani_cpu

    O = oracle
    e, _ = eng7
    sk = [O.Sketch.from_file(p.path) for p in eng7[1]]
    mean_tri, _ = e.triangle(screen=80.0, min_af=15.0)
    mean_rect, _ = e.rect([0, 1, 2, 3], [4, 5, 6], screen=80.0, min_af=15.0)
    try:
        for mode in MODES:
            e.set_estimator(mode)
            tri, _ = e.triangle(screen=80.0, min_af=15.0)
            with REF.estimator(mode):
                want = skani_cpu.triangle_edges(sk, 80.0, 15.0, 4)
            assert _fmt(tri) == {(a, b): ("%.2f" % ani, "%.2f" % afa, "%.2f" % afb) for a, b, ani, afa, afb in want}
            assert _cols(tri) == _cols(mean_tri)
            rect, _ = e.rect([0, 1, 2, 3], [4, 5, 6], screen=80.0, min_af=15.0)
            for x in rect:
                r = REF.pair(sk[int(x["a"])], sk[int(x["b"])], mode=mode)
                assert ("%.2f" % x["ani"], "%.2f" % x["af_a"], "%.2f" % x["af_b"]) == (
                    "%.2f" % (r.ani * 100), "%.2f" % (r.af_a * 100), "%.2f" % (r.af_b * 100))
            assert _cols(rect) == _cols(mean_rect)
    finally:
        e.set_estimator("mean")


@pytest.mark.gpu
def test_estimator_leaves_no_state_behind(eng7, genomes7):
    from skder_b200 import engine

    e, packed = eng7
    for mode in ("mean", "robust", "median", "mean"):
        e.set_estimator(mode)
        l0 = e.launches
        edges, _ = e.triangle(screen=80.0, min_af=15.0)
        used = e.launches - l0
    with engine.Engine(0) as fresh:
        fresh.add(packed)
        fresh.index()
        l0 = fresh.launches
        want, _ = fresh.triangle(screen=80.0, min_af=15.0)
        assert fresh.launches - l0 == used  # the mean adds no launch, after other modes or not
        assert edges.tobytes() == want.tobytes()
        # the setting is context state that survives clear(); unknown values are refused
        fresh.set_estimator("robust")
        fresh.clear()
        fresh.add(packed)
        fresh.index()
        rob, _ = fresh.triangle(screen=80.0, min_af=15.0)
        e.set_estimator("robust")
        try:
            assert rob.tobytes() == e.triangle(screen=80.0, min_af=15.0)[0].tobytes()
        finally:
            e.set_estimator("mean")
        with pytest.raises(ValueError):
            fresh.set_estimator("trimmed")
        assert fresh._L.skb_set_ani_estimator(fresh._h, 3) == -1


@pytest.mark.gpu
def test_sharded_pairs_edges_robust_equals_triangle(eng7):
    from skder_b200 import engine

    e, packed = eng7
    e.set_estimator("robust")
    try:
        full, _ = e.triangle(screen=80.0, min_af=15.0)
    finally:
        e.set_estimator("mean")
    got = []
    for first, count in [(0, 3), (3, 4)]:
        with engine.Engine(0) as e2:
            e2.set_estimator("robust")
            e2.add(packed)
            e2.index()
            e2.set_owned(first, count)
            e2.index()
            ptr, n, _ = e2.screen_triangle(80.0)
            edges, _ = e2.pairs_edges(ptr, n, owned_only=True, min_af=15.0)
            got.append(edges)
    cat = np.sort(np.concatenate(got), order=["a", "b"])
    assert cat.tobytes() == np.sort(full, order=["a", "b"]).tobytes()


def _run(script, argv, env=None):
    return subprocess.call([sys.executable, script] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **(env or {})))


@pytest.mark.gpu
def test_shim_end_to_end_equals_cpu_skani(genomes7, built_lib, tmp_path):
    from skder_b200 import daemon

    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    cpu = os.path.join(ROOT, "tests", "ani_estimators_ref.py")  # tests/oracle_skani.py with the argv's estimator
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

    out = both(["triangle", "-l", str(lst), "--min-af", "15.0", "-E", "-t", "4", "--robust"])
    assert "--robust" in open(str(out) + ".skani_b200.log").read()
    both(["dist", "--rl", str(rl), "--ql", str(ql), "--median"])
    db = tmp_path / "db"
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(db), "-t", "4"]) == 0
    q = genomes7[2]
    both(["search", q, "-d", str(db), "-t", "2", "--robust"], {"SKB_NO_DAEMON": "1"})
    try:
        for extra in ([], ["--robust"], [], ["--median"]):  # one resident server alternates between modes
            both(["search", q, "-d", str(db), "-t", "2"] + extra, {"SKB_DAEMON_IDLE": "120"})
        assert daemon.request(str(db), 0, {"op": "ping"}, timeout=5.0)["n"] == 7
    finally:
        daemon.stop_for(str(db))
    bad = tmp_path / "bad.tsv"
    assert _run(shim, ["triangle", "-l", str(lst), "-E", "--median", "--robust", "-o", str(bad)]) != 0 and not bad.exists()
