"""skani sketch files as genomes (DESIGN.md section 3): `sketch -o DB` writes DB/<basename>.sketch per input, and
triangle and dist take such files wherever they take a FASTA.  On the CPU: the parser, the descriptor names and bytes,
the CPU reference (tests/sketch_inputs_ref.py) against a hand-built database, and the refusals, which leave no output.
On the device: skb_db_load_genomes against fresh adds bit for bit, with its errors, and every sketch form of the shim
byte-identical to its FASTA form and to the reference."""
import json
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SHIM = os.path.join(ROOT, "skder_b200", "bin", "skani")
REF = os.path.join(ROOT, "tests", "sketch_inputs_ref.py")


def _run(script, argv, env=None, cwd=None):
    e = dict(os.environ, SKB_NO_DAEMON="1", **(env or {}))
    return subprocess.run([sys.executable, script] + argv, capture_output=True, env=e, cwd=cwd, timeout=900)


def _output(script, argv, extra_files=()):
    """what a command wrote -- its -o file (and the files named in extra_files), or without -o its stdout -- as bytes;
    asserts exit 0"""
    r = _run(script, argv)
    assert r.returncode == 0, (argv, r.stderr.decode())
    if "-o" not in argv:
        return r.stdout
    out = argv[argv.index("-o") + 1]
    data = [open(p, "rb").read() for p in (out,) + tuple(extra_files)]
    for p in (out,) + tuple(extra_files):
        os.unlink(p)
    return tuple(data) if extra_files else data[0]


def _lst(path, items):
    path.write_text("".join(x + "\n" for x in items))
    return str(path)


def fake_db(d, paths, names, m=1000, contigs=None):
    """a sketch database in directory d the way skb_db_save lays it out -- genome i with contigs[i] (default: one of
    1,000 bp), no seeds, no marker keys -- and its manifest; no device needed"""
    os.makedirs(d, exist_ok=True)
    n = len(paths)
    contigs = contigs or [[1000]] * n
    ctg = [x for c in contigs for x in c]
    head = (b"SKB200v1" if m == 1000 else b"SKB200v2" + struct.pack("<Q", m)) + struct.pack("<4Q", n, 0, 0, len(ctg))
    tables = (np.zeros(n + 1, "<u8").tobytes() + np.array([sum(c) for c in contigs], "<u8").tobytes()
              + np.concatenate([[0], np.cumsum([len(c) for c in contigs])]).astype("<u4").tobytes()
              + np.array(ctg, "<u4").tobytes())
    with open(os.path.join(d, "sketches.skb"), "wb") as f:
        f.write(head + tables)
    with open(os.path.join(d, "manifest.json"), "w") as f:
        json.dump({"paths": paths, "names": names}, f)


def describe(d, inputs, paths, names, per_sequence=False):
    from skder_b200 import cli, sketch_files

    sketch_files.write_all(d, inputs, paths, names, per_sequence, cli.write_atomic)


def _sketches(d):
    return {f: open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d)) if f.endswith(".sketch")}


# ---- the parser and the descriptors --------------------------------------------------------------------------------------
def test_parser_takes_sketch_forms(tmp_path):
    from skder_b200 import cli

    L = _lst(tmp_path / "l.txt", ["db/b.fa.sketch", "a.fa"])

    def inputs(*argv):
        sub, opt = cli.parse_args(list(argv))
        return cli.inputs(sub, opt)

    assert inputs("triangle", "db/c.fa.sketch", "db/a.fa.sketch", "-E") == ["db/a.fa.sketch", "db/c.fa.sketch"]
    assert inputs("triangle", "db/c.fa.sketch", "-l", L, "-E", "-i") == ["a.fa", "db/b.fa.sketch", "db/c.fa.sketch"]
    assert inputs("dist", "q.fa", "db/a.fa.sketch", "db/b.fa.sketch") == (["db/a.fa.sketch", "db/b.fa.sketch"], ["q.fa"])
    assert inputs("dist", "-q", "db/q.fa.sketch", "-r", "r.fa", "--rl", L) == (["r.fa", "db/b.fa.sketch", "a.fa"],
                                                                              ["db/q.fa.sketch"])
    assert inputs("dist", "--ql", L, "--rl", L, "-n", "2", "--qi") == (["db/b.fa.sketch", "a.fa"], ["db/b.fa.sketch", "a.fa"])
    for argv in (["sketch", "db/a.fa.sketch", "-o", "db2"], ["sketch", "a.fa", "-l", L, "-o", "db2"]):
        sub, opt = cli.parse_args(argv)
        with pytest.raises(cli.UsageError):
            cli.inputs(sub, opt)


def test_descriptor_names():
    from skder_b200.sketch_files import file_names

    got = file_names(["x/a.fa", "y/a.fa", "x/a.fa", "b.fa.gz", "z/a.fa", "w/a.fa.1", "b.fa.gz"])
    assert got == {"x/a.fa": "a.fa.sketch", "y/a.fa": "a.fa.1.sketch", "b.fa.gz": "b.fa.gz.sketch",
                   "z/a.fa": "a.fa.2.sketch", "w/a.fa.1": "a.fa.1.1.sketch"}  # the first free name
    assert list(got) == ["x/a.fa", "y/a.fa", "b.fa.gz", "z/a.fa", "w/a.fa.1"]


def test_descriptors_are_deterministic(built_lib, tmp_path):
    paths = ["g/a.fa", "h/a.fa", "g/a.fa", "b.fa"]
    names = ["na", "na2", "na", "nb"]
    for d in ("one", "two"):
        fake_db(str(tmp_path / d), paths, names)
        describe(str(tmp_path / d), paths, paths, names)
    one, two = _sketches(str(tmp_path / "one")), _sketches(str(tmp_path / "two"))
    assert one == two and sorted(one) == ["a.fa.1.sketch", "a.fa.sketch", "b.fa.sketch"]
    d = json.loads(one["a.fa.sketch"])
    assert (d["format"], d["path"], d["per_sequence"], d["ids"], d["names"]) == ("skb200-sketch-1", "g/a.fa", False, [0], ["na"])
    assert json.loads(one["b.fa.sketch"])["ids"] == [3]
    # -i: every record of the file's first occurrence
    files = ["m1.fa", "m2.fa", "m1.fa"]
    rec_paths = ["m1.fa", "m1.fa", "m2.fa", "m1.fa", "m1.fa"]
    rec_names = ["r1", "r2", "s1", "r1", "r2"]
    fake_db(str(tmp_path / "i"), rec_paths, rec_names, contigs=[[600]] * 5)
    describe(str(tmp_path / "i"), files, rec_paths, rec_names, per_sequence=True)
    s = {k: json.loads(v) for k, v in _sketches(str(tmp_path / "i")).items()}
    assert (s["m1.fa.sketch"]["ids"], s["m1.fa.sketch"]["names"], s["m1.fa.sketch"]["per_sequence"]) == ([0, 1], ["r1", "r2"], True)
    assert s["m2.fa.sketch"]["ids"] == [2]


def test_reference_rewrites_hand_built_case(oracle, built_lib, genomes7, tmp_path):
    import sketch_inputs_ref

    G = genomes7
    db, db2 = str(tmp_path / "db"), str(tmp_path / "db2")
    fake_db(db, [G[2], G[0], G[4]], ["n2", "n0", "n4"])
    describe(db, [G[2], G[0], G[4]], [G[2], G[0], G[4]], ["n2", "n0", "n4"])
    fake_db(db2, [G[5]], ["n5"], m=200)
    describe(db2, [G[5]], [G[5]], ["n5"])
    sk = {g: os.path.join(db, os.path.basename(g) + ".sketch") for g in (G[0], G[2], G[4])}
    L = _lst(tmp_path / "l.txt", [sk[G[4]], G[1]])
    tmp = str(tmp_path / "rw")
    os.makedirs(tmp)
    got = sketch_inputs_ref.rewrite(["triangle", sk[G[2]], G[3], "-l", L, "-E"], tmp)
    assert got[:3] == ["triangle", G[2], G[3]] and got[3] == "-l" and got[5:] == ["-E", "-m", "1000"]
    assert open(got[4]).read().split() == [G[4], G[1]]
    got = sketch_inputs_ref.rewrite(["dist", "-q", sk[G[0]], "-r", G[6], sk[G[2]], "-n", "2"], tmp)
    assert got == ["dist", "-q", G[0], "-r", G[6], G[2], "-n", "2", "-m", "1000"]
    assert sketch_inputs_ref.rewrite(["dist", G[1], db2 + "/" + os.path.basename(G[5]) + ".sketch", "-m", "200"], tmp) == \
        ["dist", G[1], G[5], "-m", "200"]
    from skder_b200 import cli

    for bad in (["triangle", sk[G[0]], db2 + "/" + os.path.basename(G[5]) + ".sketch", "-E"],
                ["triangle", sk[G[0]], G[1], "-E", "-m", "200"], ["triangle", sk[G[0]], G[1], "-E", "-i"],
                ["dist", "-q", sk[G[0]], "-r", G[1], "--qi"]):
        with pytest.raises(cli.UsageError):
            sketch_inputs_ref.rewrite(bad, tmp)
    # the reference's output is its FASTA form's, through the oracle
    f1, f2 = str(tmp_path / "a.tsv"), str(tmp_path / "b.tsv")
    want = _output(os.path.join(ROOT, "tests", "cli_forms_ref.py"), ["triangle", G[0], G[1], G[2], "-E", "-o", f1])
    assert want.count(b"\n") > 1
    assert _output(REF, ["triangle", sk[G[0]], G[1], sk[G[2]], "-E", "-o", f2]) == want
    assert _output(REF, ["triangle", sk[G[0]], G[1], sk[G[2]], "-E"]) == want


def test_refusals_leave_no_output(built_lib, tmp_path):
    from skder_b200 import synth

    g = str(tmp_path / "g.fa")
    synth.write_fasta(g, [b"ACGT" * 500])
    db, db_i, db_m, stale = (str(tmp_path / d) for d in ("db", "db_i", "db_m", "stale"))
    fake_db(db, [g], ["g"])
    describe(db, [g], [g], ["g"])
    fake_db(db_i, [g], ["g"])
    describe(db_i, [g], [g], ["g"], per_sequence=True)
    fake_db(db_m, [g], ["g"], m=200)
    describe(db_m, [g], [g], ["g"])
    fake_db(stale, [g], ["g"])
    describe(stale, [g], [g], ["g"])
    fake_db(stale, [g, g], ["g", "g"])  # a later sketch into the same directory: the old descriptor is stale
    S = {d: os.path.join(d, "g.fa.sketch") for d in (db, db_i, db_m, stale)}
    L = _lst(tmp_path / "l.txt", [S[db]])
    out = str(tmp_path / "o.tsv")
    cwd = tmp_path / "cwd"
    cwd.mkdir()
    cases = [
        (["triangle", S[stale], g, "-E"], b"does not belong"),
        (["dist", g, S[stale]], b"does not belong"),
        (["triangle", S[db], S[db_m], "-E"], b"UsageError"),   # two databases, two m
        (["triangle", S[db], g, "-E", "-m", "200"], b"UsageError"),
        (["dist", "-q", g, "-r", S[db_m], "-m", "1000"], b"UsageError"),
        (["triangle", S[db], g, "-E", "-i"], b"UsageError"),   # a file-mode sketch has no record sketches
        (["triangle", S[db_i], g, "-E"], b"UsageError"),      # an -i sketch on a side without -i
        (["dist", "-q", S[db], "-r", g, "--qi"], b"UsageError"),
        (["dist", "-q", g, "-r", S[db_i]], b"UsageError"),
        (["dist", "--ql", L, "-r", g, "--qi"], b"UsageError"),
    ]
    for argv, why in cases:
        r = _run(SHIM, argv + ["-o", out])
        assert r.returncode != 0 and not os.path.exists(out) and r.stdout == b"" and why in r.stderr, (argv, r.stderr)
        r = _run(SHIM, argv, cwd=str(cwd))  # the stdout form
        assert r.returncode != 0 and r.stdout == b"" and why in r.stderr, (argv, r.stderr)
    for argv in (["sketch", S[db], "-o", str(tmp_path / "db_new")], ["sketch", g, "-l", L, "-o", str(tmp_path / "db_new")]):
        r = _run(SHIM, argv)
        assert r.returncode != 0 and b"UsageError" in r.stderr and not os.path.exists(str(tmp_path / "db_new")), argv
    assert os.listdir(cwd) == []
    # the accepted pairings: a sketch's label is its recorded path, on a side of its database's mode
    from skder_b200 import cli

    descs = cli.sketch_sources([S[db_i], g], {"marker_c": 1000, "marker_c_given": False})
    assert cli.genome_unit(S[db_i], True, descs, "-i")[0] == (g, True)
    descs = cli.sketch_sources([S[db]], {"marker_c": 1000, "marker_c_given": True})
    assert cli.genome_unit(S[db], False, descs, "--qi")[0] == (g, False)


# ---- the library on the device -----------------------------------------------------------------------------------------
def _same_genomes(a, b):
    """two indexed engines hold the same genomes bit for bit: seeds, markers, contig statistics, shared markers and the
    triangle's edges"""
    n = a.n_genomes
    assert b.n_genomes == n
    for g in range(n):
        assert a.sizes(g) == b.sizes(g), g
        assert np.array_equal(a.seeds(g), b.seeds(g)), g
        assert np.array_equal(a.markers(g), b.markers(g)), g
    for x, y in zip(a.contig_stats(0, n), b.contig_stats(0, n)):
        assert np.array_equal(x, y)
    ia, ib = np.triu_indices(n, 1)
    assert np.array_equal(a.shared_markers(ia, ib), b.shared_markers(ia, ib))
    ea, _ = a.triangle(screen=80.0, min_af=15.0)
    eb, _ = b.triangle(screen=80.0, min_af=15.0)
    assert len(ea) > 0 and ea.tobytes() == eb.tobytes()


@pytest.mark.gpu
def test_load_genomes_equals_fresh_adds(built_lib, genomes7, tmp_path):
    from skder_b200 import engine
    from skder_b200._lib import SkbError

    G = genomes7
    for m in (1000, 200):
        db = str(tmp_path / ("db%d" % m))
        with engine.Engine(0) as e:
            e.set_marker_compression(m)
            e.add_fasta(G, threads=4)
            e.save(db)
        assert engine.db_info(db)[:2] == (7, m)
        pick = [5, 2, 0, 6, 3]
        with engine.Engine(0) as fresh, engine.Engine(0) as loaded:
            fresh.set_marker_compression(m)
            fresh.add_fasta([G[i] for i in pick], threads=4)
            fresh.index()
            loaded.load_genomes(db, pick)  # an empty context takes the database's m
            assert loaded.marker_compression == m
            loaded.index()
            _same_genomes(fresh, loaded)
        # mixed with FASTA adds, and one pop_last_add undoes a load
        with engine.Engine(0) as fresh, engine.Engine(0) as mixed:
            for e in (fresh, mixed):
                e.set_marker_compression(m)
            fresh.add_fasta([G[1], G[4], G[2], G[6]], threads=4)
            fresh.index()
            mixed.add_fasta([G[1]], threads=4)
            mixed.load_genomes(db, [0, 3])
            assert mixed.n_genomes == 3
            mixed.pop_last_add()
            assert mixed.n_genomes == 1
            mixed.load_genomes(db, [4, 2])
            mixed.add_fasta([G[6]], threads=4)
            mixed.index()
            _same_genomes(fresh, mixed)
    # errors
    db = str(tmp_path / "db1000")
    with engine.Engine(0) as e:
        for ids in ([7], [-1], [1, 2, 1]):  # out of range, repeated: SKB_EINVAL
            with pytest.raises(SkbError, match=r"\(-1\)"):
                e.load_genomes(db, ids)
        assert e.n_genomes == 0
        with pytest.raises(SkbError, match=r"\(-3\)"):
            e.load_genomes(str(tmp_path / "nowhere"), [0])
        e.set_marker_compression(200)
        e.add_fasta([G[0]], threads=4)
        with pytest.raises(SkbError, match=r"\(-5\)"):
            e.load_genomes(db, [1])
        assert e.n_genomes == 1
        e.load_genomes(str(tmp_path / "db200"), [1])
        assert e.n_genomes == 2


# ---- the shim on the device --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sketch_forms_equal_fasta_forms(built_lib, genomes7, tmp_path):
    from test_cli_forms import multi_fastas

    G = genomes7
    M = multi_fastas(tmp_path)
    n = [0]

    def lst(items):
        n[0] += 1
        return _lst(tmp_path / ("l%d.txt" % n[0]), items)

    dbs = {}
    for name, form in (("db", G[:5]), ("db2", G[4:]), ("db_m", ["-m", "200"] + G[:4]), ("db_i", ["-i"] + M)):
        dbs[name] = str(tmp_path / name)
        r = _run(SHIM, ["sketch"] + form + ["-o", dbs[name]])
        assert r.returncode == 0, r.stderr.decode()

    def sk(db, g):
        return os.path.join(dbs[db], os.path.basename(g) + ".sketch")

    assert sorted(_sketches(dbs["db"])) == sorted(os.path.basename(g) + ".sketch" for g in G[:5])
    f_new, f_fa = str(tmp_path / "new.tsv"), str(tmp_path / "fa.tsv")

    def check(new, fasta, matrix=False):
        """the sketch form's -o file and stdout and the CPU reference's output all equal the FASTA form's"""
        extra = (f_fa + ".af",) if matrix else ()
        want = _output(SHIM, fasta + ["-o", f_fa], extra)
        assert (want[0] if matrix else want).count(b"\n") > 2, fasta
        got = _output(SHIM, new + ["-o", f_new], (f_new + ".af",) if matrix else ())
        assert got == want, new
        if matrix:
            assert _output(REF, new + ["-o", f_new], (f_new + ".af",)) == want, new
            return
        assert _output(SHIM, new) == want, new
        assert _output(REF, new) == want, new

    all5 = [sk("db", g) for g in G[:5]]
    for extra in (["-E"], ["-E", "--ci"], ["-E", "--detailed"], ["-E", "--median", "-s", "85"]):
        check(["triangle", *all5] + extra, ["triangle", *G[:5]] + extra)
    for extra in (["--full-matrix"], ["--full-matrix", "--distance"]):
        check(["triangle", *all5[::-1]] + extra, ["triangle", *G[:5]] + extra, matrix=True)
    check(["triangle", *[sk("db_m", g) for g in G[:4]], "-E"], ["triangle", *G[:4], "-E", "-m", "200"])
    check(["triangle", *[sk("db_i", p) for p in M], "-E", "-i"], ["triangle", *M, "-E", "-i"])
    # mixed FASTA and sketch arguments, lists holding sketches, a label named both ways, two databases
    check(["triangle", G[6], sk("db", G[3]), "-l", lst([sk("db", G[0]), G[5], G[3]]), "-E"],
          ["triangle", G[6], G[3], G[0], G[5], "-E"])
    check(["triangle", sk("db", G[1]), sk("db2", G[6]), sk("db2", G[4]), sk("db", G[4]), "-E", "--ci"],
          ["triangle", G[1], G[6], G[4], "-E", "--ci"])
    # dist
    check(["dist", G[6], *all5], ["dist", G[6], *G[:5]])
    check(["dist", "-q", sk("db", G[0]), G[5], "-r", *all5[1:], G[6], "-n", "2"],
          ["dist", "-q", G[0], G[5], "-r", *G[1:5], G[6], "-n", "2"])
    check(["dist", "--ql", lst([sk("db", G[1]), G[6]]), "--rl", lst([sk("db2", G[5]), sk("db", G[2]), G[1]]), "--detailed"],
          ["dist", "--ql", lst([G[1], G[6]]), "--rl", lst([G[5], G[2], G[1]]), "--detailed"])
    check(["dist", "-q", sk("db", G[2]), sk("db2", G[6]), "-r", G[2], sk("db", G[3]), "--median"],
          ["dist", "-q", G[2], G[6], "-r", G[2], G[3], "--median"])
    check(["dist", "-q", sk("db_i", M[0]), "-r", sk("db_i", M[1]), M[2], "--qi", "--ri", "-n", "2"],
          ["dist", "-q", M[0], "-r", M[1], M[2], "--qi", "--ri", "-n", "2"])
    check(["dist", "-q", sk("db_i", M[0]), "-r", M[0], M[1], "--qi"], ["dist", "-q", M[0], "-r", M[0], M[1], "--qi"])
    check(["dist", sk("db_m", G[0]), sk("db_m", G[1]), G[2]], ["dist", G[0], G[1], G[2], "-m", "200"])
