"""skani's `triangle --full-matrix [--distance]` (DESIGN.md section 3): the parser's forms and refusals, refusals that
leave no file, the CPU reference (tests/matrix_ref.py) against a numpy restatement from the oracle's edge list, and on
the device skb_write_matrix's exact `%.2f` text, the shim byte-identical to the reference and to its own -E TSV, the
state and argument errors, and a few hundred genomes rendered in many row blocks."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import matrix_ref  # noqa: E402

SEED = 20261025
SHIM = os.path.join(ROOT, "skder_b200", "bin", "skani")
REF = os.path.join(ROOT, "tests", "matrix_ref.py")


def _run(script, argv, env=None, cwd=None):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, script] + argv, capture_output=True, env=e, cwd=cwd, timeout=900)


def _outputs(script, argv, cwd, env=None):
    """(ANI file bytes, AF file bytes) of a command: -o OUT and OUT.af, or without -o stdout and cwd/skani_matrix.af"""
    targets = [argv[argv.index("-o") + 1]] if "-o" in argv else []
    targets.append(targets[0] + ".af" if targets else os.path.join(cwd, "skani_matrix.af"))
    for t in targets:
        if os.path.exists(t):
            os.unlink(t)
    r = _run(script, argv, env, cwd)
    assert r.returncode == 0, (argv, r.stderr.decode())
    files = [open(t, "rb").read() for t in targets]
    if "-o" in argv:
        assert r.stdout == b"", argv
        return files[0], files[1]
    return r.stdout, files[0]


def _text(v):
    """`%.2f` of hundredths"""
    return ("-" if v < 0 else "") + "%d.%02d" % divmod(abs(int(v)), 100)


def render(n, labels, edges, kind):
    """the matrix file of an EDGE_DTYPE-like list, formatted by Python"""
    a, b = edges["a"].astype(np.int64), edges["b"].astype(np.int64)
    m = np.full((n, n), "100.00" if kind == "distance" else "0.00", object)
    if kind == "af":
        m[a, b] = ["%.2f" % x for x in edges["af_a"].tolist()]
        m[b, a] = ["%.2f" % x for x in edges["af_b"].tolist()]
    else:
        t = ["%.2f" % x for x in edges["ani"].tolist()]
        if kind == "distance":
            t = [_text(10000 - matrix_ref.cents(x)) for x in t]
        m[a, b] = m[b, a] = t
    np.fill_diagonal(m, "0.00" if kind == "distance" else "100.00")
    return ("%d\n" % n + "".join(lb + "".join("\t" + x for x in row) + "\n" for lb, row in zip(labels, m.tolist()))).encode()


# ---- the parser ---------------------------------------------------------------------------------------------------------
def test_parser_forms_and_refusals(tmp_path):
    from skder_b200 import cli

    L = str(tmp_path / "l.txt")
    with open(L, "w") as f:
        f.write("b.fa\na.fa\n")
    for argv in (["triangle", "b.fa", "a.fa", "--full-matrix"], ["triangle", "-l", L, "--full-matrix", "-o", "o"],
                 ["triangle", "a.fa", "--full-matrix", "--distance", "-s", "85", "--min-af", "30", "-m", "200", "-t", "4"],
                 ["triangle", "a.fa", "-l", L, "--distance", "--full-matrix", "--median"],
                 ["triangle", "a.fa", "--full-matrix", "--robust", "-i"]):
        sub, opt = cli.parse_args(argv)
        assert sub == "triangle" and opt["full_matrix"] and not opt["edge_list"], argv
        assert opt["distance"] == ("--distance" in argv), argv
        assert cli.inputs(sub, opt) == (["a.fa", "b.fa"] if "b.fa" in argv or L in argv else ["a.fa"])
    _, opt = cli.parse_args(["triangle", "a.fa", "-E"])
    assert not opt["full_matrix"] and not opt["distance"]
    bad = ["triangle a.fa --full-matrix -E", "triangle a.fa -E --full-matrix -o o", "triangle a.fa --distance",
           "triangle a.fa -E --distance", "dist a.fa b.fa --full-matrix", "dist -q a.fa -r b.fa --distance",
           "search a.fa -d db --full-matrix", "sketch a.fa -o db --full-matrix", "sketch a.fa -o db --distance",
           "triangle a.fa --full-matrix --ci", "triangle a.fa --full-matrix --detailed -o o",
           "triangle a.fa --full-matrix --diagonal", "triangle a.fa -E --diagonal", "triangle a.fa --diagonal",
           "triangle a.fa b.fa", "triangle -l L -o o", "triangle a.fa --full-matrix -c 30"]
    for argv in bad:
        with pytest.raises(cli.UsageError):
            cli.parse_args(argv.split())
    with pytest.raises(cli.UsageError, match="use -E or --full-matrix"):
        cli.parse_args(["triangle", "a.fa", "b.fa"])


def test_refusals_leave_no_output(tmp_path):
    out = tmp_path / "o.txt"
    cwd = tmp_path / "cwd"
    cwd.mkdir()
    for argv in (["triangle", "a.fa", "b.fa", "--full-matrix", "-E"], ["triangle", "a.fa", "b.fa", "--distance"],
                 ["triangle", "a.fa", "b.fa", "--full-matrix", "--ci"], ["triangle", "a.fa", "--full-matrix", "--detailed"],
                 ["dist", "a.fa", "b.fa", "--full-matrix"], ["triangle", "a.fa", "b.fa", "--full-matrix", "--diagonal"],
                 ["triangle", "a.fa", "b.fa"]):
        r = _run(SHIM, argv + ["-o", str(out)], {"SKB_NO_DAEMON": "1"}, cwd=str(cwd))
        assert r.returncode != 0 and r.stdout == b"", argv
        assert not out.exists() and not (tmp_path / "o.txt.af").exists(), argv
        r = _run(SHIM, argv, {"SKB_NO_DAEMON": "1"}, cwd=str(cwd))  # the stdout form
        assert r.returncode != 0 and r.stdout == b"" and b"UsageError" in r.stderr, argv
        assert os.listdir(cwd) == [], argv
    assert sorted(os.listdir(tmp_path)) == ["cwd", "o.txt.skani_b200.log"]  # the failure note beside -o, nothing else


# ---- the CPU reference against a restatement from the oracle's edge list ------------------------------------------------
def _restated(labels, sketches, screen, min_af, distance):
    """(ANI or distance file, AF file): the oracle's edges filled into dense numpy arrays"""
    from oracle import skani_cpu

    n = len(sketches)
    e = skani_cpu.triangle_edges(sketches, screen, min_af, 4)
    edges = np.zeros(len(e), [("a", "<u4"), ("b", "<u4"), ("ani", "<f8"), ("af_a", "<f8"), ("af_b", "<f8")])
    for i, row in enumerate(e):
        edges[i] = row
    return render(n, labels, edges, "distance" if distance else "ani"), render(n, labels, edges, "af")


def multi_fastas(d):
    """two multi-record files over two clades of 20 kb sequences, one record under 500 bp, and a one-record file;
    returns (paths, [(header, sequence)] of the kept records in triangle order)"""
    from skder_b200 import synth

    cl = [[g[0] for g in synth.one_clade(c, 4, 20_000, SEED, d_lo=0.001, d_hi=0.01, max_contigs=1)] for c in range(2)]
    files = {"m1.fa": [cl[0][0], cl[1][0], b"ACGT" * 100, cl[0][1]], "m2.fa": [cl[1][1], cl[0][2], cl[1][2]],
             "m3.fa": [cl[0][3]]}
    paths, recs = [], []
    for name, seqs in files.items():
        paths.append(str(d / name))
        synth.write_fasta(paths[-1], seqs, name=name.split(".")[0])
        recs += [("%s_%d" % (name.split(".")[0], i + 1), s) for i, s in enumerate(seqs) if len(s) >= 500]
    return paths, recs


def test_reference_equals_restatement(oracle, genomes7, tmp_path):
    G = genomes7
    sk = [oracle.Sketch.from_file(p) for p in G]
    out = str(tmp_path / "m.txt")
    for extra, screen, min_af in (([], 80.0, 15.0), (["--distance"], 80.0, 15.0), (["-s", "85", "--distance"], 85.0, 15.0),
                                  (["--min-af", "90"], 80.0, 90.0)):
        want = _restated(G, sk, screen, min_af, "--distance" in extra)
        assert want[0].count(b"\t0.00" if "--distance" not in extra else b"\t100.00") < 42
        argv = ["triangle", *G[::-1], "--full-matrix"] + extra
        assert _outputs(REF, argv + ["-o", out], str(tmp_path)) == want, extra
        assert _outputs(REF, argv, str(tmp_path)) == want, extra
    # -i: every kept record is a genome, labelled by its header
    paths, recs = multi_fastas(tmp_path)
    sk = [oracle.Sketch.from_contigs([s]) for _, s in recs]
    for extra in ([], ["--distance"]):
        want = _restated([h for h, _ in recs], sk, 80.0, 15.0, bool(extra))
        assert _outputs(REF, ["triangle", *paths, "-i", "--full-matrix", "-o", out] + extra, str(tmp_path)) == want


# ---- on the device ------------------------------------------------------------------------------------------------------
def _crafted_values():
    """0, 100, ties of the third decimal, both neighbours of every k/100 +- 0.005, and 10^6 seeded uniform doubles"""
    v = [0.0, 100.0, 0.125, 2.675, 1.005, 99.995, 0.005, 0.015, 50.0, 99.99]
    for k in range(10001):
        for x in (k / 100 + 0.005, k / 100 - 0.005, k / 100):
            v += [x, np.nextafter(x, -np.inf), np.nextafter(x, np.inf)]
    v = np.array(v)
    v = v[(v >= 0) & (v <= 100)]
    return np.concatenate([v, np.random.default_rng(SEED).uniform(0.0, 100.0, 1_000_000)])


@pytest.mark.gpu
def test_exact_formatting_in_many_blocks(built_lib, tmp_path, monkeypatch):
    from skder_b200 import engine

    vals = _crafted_values()
    n = 1500  # 1,124,250 pairs; rows of 1,500 cells are longer than one CTA tile of 1,024
    a, b = np.triu_indices(n, 1)
    rng = np.random.default_rng(SEED + 1)
    keep = np.sort(rng.choice(len(a), len(vals), replace=False))
    edges = np.zeros(len(keep), engine.EDGE_DTYPE)
    edges["a"], edges["b"] = a[keep], b[keep]
    for col in ("ani", "af_a", "af_b"):
        edges[col] = rng.permutation(vals)
    labels = ["g%04d é" % i for i in range(n)]
    monkeypatch.setenv("SKB_MATRIX_BLOCK_MB", "2")  # ~ 120 rows a block: 13 blocks
    with engine.Engine(0) as eng:
        for kind in ("ani", "distance", "af"):
            p = str(tmp_path / kind)
            eng.write_matrix(p, labels, kind, edges)
            assert open(p, "rb").read() == render(n, labels, edges, kind), kind


@pytest.mark.gpu
def test_shim_equals_reference(built_lib, genomes7, tmp_path):
    from skder_b200 import cli

    G = genomes7
    paths, _ = multi_fastas(tmp_path)
    L = str(tmp_path / "l.txt")
    with open(L, "w") as f:
        f.write("".join(p + "\n" for p in (G[0], G[5], G[2])))
    cwd = str(tmp_path)
    out = str(tmp_path / "m.txt")

    def check(argv, env=None):
        want = _outputs(REF, argv + ["-o", out], cwd)
        assert _outputs(SHIM, argv + ["-o", out], cwd, env) == want, argv
        assert _outputs(SHIM, argv, cwd, env) == want, argv
        # every off-diagonal cell is the column text of the same run's -E row
        e_argv = [a for a in argv if a not in ("--full-matrix", "--distance")] + ["-E", "-o", out + ".tsv"]
        r = _run(SHIM, e_argv, env, cwd)
        assert r.returncode == 0, r.stderr.decode()
        _, opt = cli.parse_args(argv)
        labels, keys = matrix_ref.genomes(opt)
        got = tuple(x.encode() for x in matrix_ref.matrices(open(out + ".tsv").read(), labels, keys, opt["per_seq"],
                                                             opt["distance"]))
        assert got == want, argv
        return want

    for extra in ([], ["--distance"], ["-s", "85", "--min-af", "30"], ["-m", "200", "--distance"], ["--median"]):
        w = check(["triangle", G[6], G[1], "-l", L, "--full-matrix", "-t", "4"] + extra)
        assert w[0].startswith(b"5\n") and w[1].startswith(b"5\n")
        check(["triangle", "-l", L, "--full-matrix"] + extra, {"SKB_MATRIX_BLOCK_MB": "1"})
    for extra in ([], ["--distance"]):
        w = check(["triangle", *paths, "-i", "--full-matrix"] + extra)
        assert w[0].startswith(b"7\nm1_1\t")


@pytest.mark.gpu
def test_edge_cases(built_lib, tmp_path):
    from skder_b200 import engine, synth

    g = str(tmp_path / "g.fa")
    h = str(tmp_path / "h.fa")
    rng = np.random.default_rng(SEED)
    synth.write_fasta(g, [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 20_000)].tobytes()])
    synth.write_fasta(h, [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 20_000)].tobytes()])
    out = str(tmp_path / "m.txt")
    assert _outputs(SHIM, ["triangle", g, "--full-matrix", "-o", out], str(tmp_path)) == (("1\n%s\t100.00\n" % g).encode(),) * 2
    assert _outputs(SHIM, ["triangle", h, g, "--full-matrix", "--distance", "-o", out], str(tmp_path)) == \
        (("2\n%s\t0.00\t100.00\n%s\t100.00\t0.00\n" % (g, h)).encode(), ("2\n%s\t100.00\t0.00\n%s\t0.00\t100.00\n" % (g, h)).encode())
    assert sorted(os.listdir(tmp_path)) == ["g.fa", "h.fa", "m.txt", "m.txt.af", "m.txt.skani_b200.log"]

    gens = [engine.pack_contigs(c) for c in synth.one_clade(0, 4, 60_000, SEED, d_lo=0.005, d_hi=0.02, max_contigs=2)]
    labels = ["a", "b", "c", "d"]
    p = str(tmp_path / "x")
    with engine.Engine(0) as eng:
        eng.add(gens)
        eng.index()
        with pytest.raises(engine.SkbError, match=r"\(-5\)"):  # no triangle yet
            eng.write_matrix(p, labels)
        edges, _ = eng.triangle()
        assert len(edges) == 6
        eng.write_matrix(p, labels)
        assert open(p, "rb").read() == render(4, labels, edges, "ani")
        with pytest.raises(engine.SkbError, match=r"\(-1\)"):  # n_genomes is not the context's
            eng.write_matrix(p, labels[:3])
        eng.rect([0, 1], [2, 3])
        with pytest.raises(engine.SkbError, match=r"\(-5\)"):
            eng.write_matrix(p, labels)
        eng.triangle(part=0, n_parts=2)
        with pytest.raises(engine.SkbError, match=r"\(-5\)"):
            eng.write_matrix(p, labels)
        eng.triangle()
        eng.write_matrix(p, labels, "af")
        eng.add(gens[:1])
        with pytest.raises(engine.SkbError, match=r"\(-5\)"):
            eng.write_matrix(p, labels + ["e"])
        eng.pop_last_add()
        with pytest.raises(engine.SkbError, match=r"\(-5\)"):
            eng.write_matrix(p, labels)
        # host lists: unsorted, duplicated, out of range, a value outside [0, 100]
        good = edges.copy()
        eng.write_matrix(p, labels, "distance", good)
        assert open(p, "rb").read() == render(4, labels, edges, "distance")
        bad = [good[::-1], np.concatenate([good[:2], good[1:]]), good.copy(), good.copy(), good.copy(), good.copy()]
        bad[2]["b"][0] = 4
        bad[3]["b"][0] = bad[3]["a"][0]
        bad[4]["af_b"][1] = 100.0001
        bad[5]["ani"][2] = np.nan
        for e in bad:
            with pytest.raises(engine.SkbError, match=r"\(-1\)"):
                eng.write_matrix(p, labels, "ani", e)
        with pytest.raises(engine.SkbError, match=r"\(-1\)"):
            eng._ck(eng._L.skb_write_matrix(eng._h, p.encode(), 3, None, 0, 4, b"abcd",
                                            np.arange(5, dtype=np.int64).ctypes.data), "skb_write_matrix")


@pytest.mark.gpu
def test_scale_in_many_blocks(built_lib, tmp_path, monkeypatch):
    from skder_b200 import engine, synth

    gens = [engine.pack_contigs(c) for k in range(40)
            for c in synth.one_clade(k, 8, 40_000, SEED, d_lo=0.002, d_hi=0.06, max_contigs=3)]
    n = len(gens)
    labels = ["clade%02d/member%d.fa" % (i // 8, i % 8) for i in range(n)]
    monkeypatch.setenv("SKB_MATRIX_BLOCK_MB", "1")
    with engine.Engine(0) as eng:
        eng.add(gens)
        eng.index()
        edges, _ = eng.triangle(screen=80.0, min_af=15.0)
        assert 0 < len(edges) <= 40 * 28
        for kind in ("ani", "distance", "af"):
            p = str(tmp_path / kind)
            eng.write_matrix(p, labels, kind)
            assert open(p, "rb").read() == render(n, labels, edges, kind), kind
