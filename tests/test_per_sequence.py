"""skani's per-sequence mode (-i, --qi, --ri; DESIGN.md section 3): the shim's parser, the packer's record names, the CPU
reference (tests/per_sequence_ref.py) against a restatement with one FASTA per record, the daemon's refusal path, and on
the device: skb_add_sequences against every record added as a genome of its own, bit for bit (sketches, then the edges
of triangle, rect and search in every ANI mode), and the shim end to end against the CPU reference."""
import gzip
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 20261023
SHIM = os.path.join(ROOT, "skder_b200", "bin", "skani")
CPU = os.path.join(ROOT, "tests", "per_sequence_ref.py")


def _run(script, argv, env=None):
    return subprocess.call([sys.executable, script] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **(env or {})))


def _write(path, recs, width=70):
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "wt") as f:
        for name, seq in recs:
            seq = seq.decode() if isinstance(seq, bytes) else seq
            f.write(">%s\n" % name)
            for i in range(0, len(seq), width):
                f.write(seq[i:i + width] + "\n")


def multi_fastas(d):
    """four multi-record files over two clades of 20-24 kb sequences, with records under 500 bp, a duplicate header, a
    gzip file, a one-record file and a file with no record of 500 bp"""
    from skder_b200 import synth

    rng = np.random.default_rng(SEED)
    clades = [[g[0] for g in synth.one_clade(c, 5, 20_000, SEED, d_lo=0.0005, d_hi=0.004, max_contigs=1)] for c in range(2)]

    def short(n):
        return "".join("ACGT"[x] for x in rng.integers(0, 4, n))

    files = {
        "a.fa": [("a1 first", clades[0][0]), ("tiny", short(300)), ("a2", clades[1][0]), ("a3", clades[0][1])],
        "b.fa.gz": [("dup", clades[0][2]), ("dup", clades[1][1]), ("b3", short(499)), ("b4", clades[1][2])],
        "c.fa": [("c1 only", clades[0][3])],
        "d.fa": [("d1", short(200)), ("d2", short(450))],
        "e.fa": [("e1", clades[1][3]), ("e2", clades[0][4]), ("e3", short(500))],
    }
    paths = {}
    for name, recs in files.items():
        paths[name] = str(d / name)
        _write(paths[name], recs)
    return paths, files


# ---- the parser ---------------------------------------------------------------------------------------------------------
def test_parser_accepts_and_refuses():
    from skder_b200 import cli

    ok = {("triangle", "-l", "l", "-E", "-o", "o", "-i"): "per_seq", ("sketch", "-l", "l", "-o", "o", "-i"): "per_seq",
          ("dist", "--rl", "r", "--ql", "q", "-o", "o", "--qi"): "query_per_seq",
          ("dist", "--rl", "r", "--ql", "q", "-o", "o", "--ri"): "ref_per_seq",
          ("search", "a.fa", "-d", "db", "-o", "o", "--qi"): "query_per_seq"}
    for argv, k in ok.items():
        _, opt = cli.parse_args(list(argv))
        assert opt[k] and sum(opt[x] for x in ("per_seq", "query_per_seq", "ref_per_seq")) == 1, argv
    _, opt = cli.parse_args(["dist", "--rl", "r", "--ql", "q", "-o", "o", "--qi", "--ri", "-n", "2", "--ci"])
    assert opt["query_per_seq"] and opt["ref_per_seq"] and opt["max_results"] == 2
    _, opt = cli.parse_args(["triangle", "-l", "l", "-E", "-o", "o"])
    assert not (opt["per_seq"] or opt["query_per_seq"] or opt["ref_per_seq"])
    for argv in (["dist", "--rl", "r", "--ql", "q", "-o", "o", "-i"], ["search", "a.fa", "-d", "db", "-o", "o", "-i"],
                 ["triangle", "-l", "l", "-E", "-o", "o", "--qi"], ["sketch", "-l", "l", "-o", "o", "--qi"],
                 ["triangle", "-l", "l", "-E", "-o", "o", "--ri"], ["sketch", "-l", "l", "-o", "o", "--ri"],
                 ["search", "a.fa", "-d", "db", "-o", "o", "--ri"], ["triangle", "-l", "l", "-o", "o", "-i"],
                 ["search", "a.fa", "-d", "db", "-o", "o", "--qi", "-m", "200"]):
        with pytest.raises(cli.UsageError):
            cli.parse_args(argv)


def test_refusals_leave_no_output(tmp_path):
    out = tmp_path / "o.tsv"
    for argv in (["dist", "--rl", "r", "--ql", "q", "-i"], ["search", "a.fa", "-d", "db", "-i"],
                 ["triangle", "-l", "l", "-E", "--qi"], ["sketch", "-l", "l", "--ri"]):
        assert _run(SHIM, argv + ["-o", str(out)], {"SKB_NO_DAEMON": "1"}) != 0 and not out.exists(), argv


# ---- the packer ---------------------------------------------------------------------------------------------------------
def _headers(path, min_len=500):
    """kept headers, restated: records whose sequence (blanks dropped) has at least min_len bases"""
    data = (gzip.open if path.endswith(".gz") else open)(path, "rb").read().decode()
    out = []
    for rec in data.split("\n>"):
        lines = rec.lstrip(">").split("\n")
        if sum(len(x.strip()) for x in lines[1:]) >= min_len:
            out.append(lines[0].rstrip("\r"))
    return out


def test_packer_contig_names(genomes7, tmp_path):
    from skder_b200 import engine

    paths, _ = multi_fastas(tmp_path)
    for p in genomes7 + list(paths.values()):
        packed = engine.pack_fasta(p)
        assert packed.contig_names == _headers(p), p
        assert len(packed.contig_names) == packed.n_contigs
        assert packed.first_name == (packed.contig_names[0] if packed.n_contigs else "")
    assert engine.pack_fasta(paths["b.fa.gz"]).contig_names == ["dup", "dup", "b4"]
    assert engine.pack_fasta(paths["d.fa"]).contig_names == []
    many = engine.pack_fasta_many(genomes7[:3] + [paths["a.fa"]], threads=2)
    assert [m.contig_names for m in many] == [_headers(p) for p in genomes7[:3] + [paths["a.fa"]]]
    assert engine.pack_contigs(["ACGT" * 200]).contig_names == []


# ---- the CPU reference against a restatement ----------------------------------------------------------------------------
class Restated:
    """every kept record written to its own one-record FASTA, numbered in genome order"""

    def __init__(self, d, paths):
        import per_sequence_ref

        self.d = d
        self.files = {}  # (path, k) -> record file
        self.back = {}  # record file -> (path, header)
        d.mkdir(exist_ok=True)
        for path in sorted(paths):
            for k, (name, seq) in enumerate(per_sequence_ref.records(path)):
                f = str(d / ("r%05d.fa" % len(self.back)))
                _write(f, [(name, seq.decode())])
                self.files[(path, k)] = f
                self.back[f] = (path, name)

    def split(self, path):
        return [self.files[(path, k)] for k in range(len([1 for p, _ in self.files if p == path]))]

    def relabel(self, text):
        lines = text.splitlines(keepends=True)
        out = [lines[0]]
        for ln in lines[1:]:
            t = ln.rstrip("\n").split("\t")
            for col, ncol in ((0, 5), (1, 6)):
                if t[col] in self.back:
                    t[col], t[ncol] = self.back[t[col]]
            out.append("\t".join(t) + "\n")
        return "".join(out)


def _lst(path, items):
    path.write_text("".join(x + "\n" for x in items))
    return str(path)


def test_cpu_reference_against_restatement(oracle, tmp_path):
    import search_queries_ref

    paths, _ = multi_fastas(tmp_path)
    P = [paths[k] for k in ("a.fa", "b.fa.gz", "c.fa", "d.fa", "e.fa")]
    rs = Restated(tmp_path / "rec", P)
    one = str(tmp_path / "one.tsv")

    def restated(argv):
        assert search_queries_ref.main(argv + ["-o", one]) == 0, argv
        return rs.relabel(open(one).read())

    def ref(argv):
        out = str(tmp_path / "ref.tsv")
        assert _run(CPU, argv + ["-o", out]) == 0, argv
        return open(out).read()

    # triangle -i: genomes in (sorted path, record) order; the record files are numbered that way
    want = restated(["triangle", "-l", _lst(tmp_path / "t.txt", [f for p in sorted(P) for f in rs.split(p)]), "-E"])
    got = ref(["triangle", "-l", _lst(tmp_path / "l.txt", P[::-1] + P[:1]), "-E", "-i"])
    assert got == want and len(got.splitlines()) > 5
    assert "\ta1 first\t" in got and "\tdup\t" in got
    # dist: --qi, --ri, both, with -n
    R, Q = [P[0], P[2], P[4]], [P[1], P[0], P[3]]
    rl, ql = _lst(tmp_path / "rl.txt", R), _lst(tmp_path / "ql.txt", Q)
    for qi, ri in ((True, False), (False, True), (True, True)):
        rside = [f for p in R for f in (rs.split(p) if ri else [p])]
        qside = [f for p in Q for f in (rs.split(p) if qi else [p])]
        for n in ([], ["-n", "2"]):
            flags = (["--qi"] if qi else []) + (["--ri"] if ri else [])
            want = restated(["dist", "--rl", _lst(tmp_path / "rr.txt", rside), "--ql", _lst(tmp_path / "rq.txt", qside)] + n)
            got = ref(["dist", "--rl", rl, "--ql", ql] + flags + n)
            assert got == want, (qi, ri, n)
            assert len(got.splitlines()) > 3
    # sketch -i, then search --qi against it
    db = str(tmp_path / "db")
    assert _run(CPU, ["sketch", "-l", _lst(tmp_path / "s.txt", [P[0], P[1], P[2]]), "-o", db, "-i"]) == 0
    man = json.load(open(os.path.join(db, "manifest.json")))
    assert man["paths"] == [P[0]] * 3 + [P[1]] * 3 + [P[2]]
    assert man["names"] == ["a1 first", "a2", "a3", "dup", "dup", "b4", "c1 only"]
    rdb = str(tmp_path / "rdb")
    assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"),
                ["sketch", "-l", _lst(tmp_path / "rs.txt", [f for p in (P[0], P[1], P[2]) for f in rs.split(p)]),
                 "-o", rdb]) == 0
    for n in ([], ["-n", "1"]):
        want = restated(["search", "-d", rdb, "--ql", _lst(tmp_path / "sq.txt", rs.split(P[4]) + rs.split(P[0]))] + n)
        got = ref(["search", P[4], "-d", db, "--ql", _lst(tmp_path / "q2.txt", [P[0]]), "--qi"] + n)
        assert got == want, n
        assert len(got.splitlines()) > 3


# ---- the daemon ---------------------------------------------------------------------------------------------------------
def test_unknown_op_server_is_replaced_never_answers_whole_file(tmp_path):
    """A server predating --qi refuses "search_records" as an unknown op: the shim stops it and starts one from this
    tree (which, without a GPU, never comes up: the call then fails without output).  The whole-file op is never sent."""
    from multiprocessing.connection import Listener

    from skder_b200 import daemon

    db = tmp_path / "db"
    db.mkdir()
    run_dir = tempfile.mkdtemp(prefix="skb-", dir="/tmp")
    env = dict(os.environ, SKB_DAEMON_DIR=run_dir, SKB_DEVICE="0", PYTHONPATH=ROOT, SKB_DAEMON_START_TIMEOUT="3",
               CUDA_VISIBLE_DEVICES="")
    env.pop("SKB_NO_DAEMON", None)
    os.environ["SKB_DAEMON_DIR"] = run_dir
    try:
        sock = daemon.socket_path(str(db), 0)
    finally:
        os.environ.pop("SKB_DAEMON_DIR", None)
    key = b"k" * 32
    with open(daemon._key_path(str(db), 0), "wb") as f:
        f.write(key)
    seen = []

    def serve():  # an old server: knows search, ping and stop
        with Listener(sock, family="AF_UNIX", authkey=key) as ls:
            while True:
                with ls.accept() as conn:
                    msg = json.loads(conn.recv_bytes().decode())
                    seen.append(msg["op"])
                    if msg["op"] == "search":
                        with open(msg["out"], "w") as f:
                            f.write("whole-file rows\n")
                        conn.send_bytes(json.dumps({"ok": True}).encode())
                    elif msg["op"] in ("ping", "stop"):
                        conn.send_bytes(json.dumps({"ok": True}).encode())
                        if msg["op"] == "stop":
                            break
                    else:
                        conn.send_bytes(json.dumps({"ok": False, "error": "unknown op"}).encode())

    th = threading.Thread(target=serve, daemon=True)
    th.start()
    for _ in range(200):
        if os.path.exists(sock):
            break
        time.sleep(0.01)
    out = tmp_path / "out.tsv"
    try:
        r = subprocess.run([sys.executable, "-m", "skder_b200.cli", "search", "q1.fa", "--qi", "-d", str(db), "-o",
                            str(out)], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=120)
        th.join(timeout=10)
    finally:
        shutil.rmtree(run_dir, ignore_errors=True)
    assert seen[:2] == ["search_records", "stop"] and "search" not in seen, seen
    assert r.returncode != 0 and not out.exists()


# ---- on the device ------------------------------------------------------------------------------------------------------
def _bits(a):
    if a.dtype.names is None:
        return np.ascontiguousarray(a).tobytes()
    return b"".join(np.ascontiguousarray(a[k]).tobytes() for k in a.dtype.names)


def _records_of(packed_paths):
    import per_sequence_ref

    return [seq for p in packed_paths for _, seq in per_sequence_ref.records(p)]


def _random_records(path, n, lo, hi, seed):
    rng = np.random.default_rng(seed)
    recs = []
    for i in range(n):
        L = int(rng.integers(lo, hi + 1))
        recs.append(("s%d" % i, "".join("ACGT"[x] for x in rng.integers(0, 4, L))))
    _write(path, recs)
    return path


def _assert_same_sketches(ea, eb, n):
    assert ea.n_genomes == eb.n_genomes == n
    for e in (ea, eb):  # the read-back of sizes and markers needs the index
        e.index()
    for g in range(n):
        assert ea.sizes(g) == eb.sizes(g), g
        assert np.array_equal(ea.seeds(g), eb.seeds(g)), g
        assert np.array_equal(ea.markers(g), eb.markers(g)), g
    for x, y in zip(ea.contig_stats(0, n), eb.contig_stats(0, n)):
        assert np.array_equal(x, y)


@pytest.mark.gpu
def test_sketch_parity(built_lib, genomes7, tmp_path):
    from skder_b200 import engine

    paths, _ = multi_fastas(tmp_path)
    many = _random_records(str(tmp_path / "many.fa"), 3000, 500, 3000, SEED)
    big = _random_records(str(tmp_path / "big.fa"), 4, 40_000, 70_000, SEED + 1)  # several tiles per record
    sets = {"genomes7": genomes7, "many": [many], "big": [big, paths["d.fa"], paths["a.fa"]],
            "multi": list(paths.values())}
    for name, files in sets.items():
        packed = engine.pack_fasta_many(files, threads=4)
        recs = _records_of(files)
        with engine.Engine(0) as ea, engine.Engine(0) as eb:
            ea.add(packed, per_sequence=True)
            eb.add([engine.pack_contigs([r]) for r in recs])
            _assert_same_sketches(ea, eb, len(recs))
    # a file without kept records adds nothing; mixed calls in one context; one pop undoes one add_sequences
    packed = engine.pack_fasta_many([paths["a.fa"], paths["b.fa.gz"], paths["d.fa"], paths["e.fa"]], threads=2)
    with engine.Engine(0) as ea, engine.Engine(0) as eb:
        ea.add([packed[2]], per_sequence=True)
        assert ea.n_genomes == 0
        ea.add(packed[:2])
        ea.add(packed, per_sequence=True)
        ea.add(packed[3:])
        assert ea.n_genomes == 2 + 9 + 1
        ea.pop_last_add()
        ea.pop_last_add()
        assert ea.n_genomes == 2
        ea.add(packed, per_sequence=True)
        ea.add(packed[3:])
        eb.add(packed[:2])
        eb.add([engine.pack_contigs([r]) for r in _records_of([paths[k] for k in ("a.fa", "b.fa.gz", "d.fa", "e.fa")])])
        eb.add(packed[3:])
        _assert_same_sketches(ea, eb, eb.n_genomes)


@pytest.mark.gpu
def test_engine_edges_equal_separate_genomes(built_lib, tmp_path):
    from skder_b200 import engine

    paths, _ = multi_fastas(tmp_path)
    files = [paths[k] for k in ("a.fa", "b.fa.gz", "c.fa", "d.fa", "e.fa")]
    packed = engine.pack_fasta_many(files, threads=4)
    recs = _records_of(files)
    n = len(recs)
    refs, queries = list(range(0, n, 2)), list(range(1, n, 2))
    for m in (1000, 200):
        with engine.Engine(0) as ea, engine.Engine(0) as eb:
            for e in (ea, eb):
                e.set_marker_compression(m)
            ea.add(packed, per_sequence=True)
            eb.add([engine.pack_contigs([r]) for r in recs])
            for e in (ea, eb):
                e.index()
            for mode in ("mean", "median", "robust", "ci", "detailed"):
                res = []
                for e in (ea, eb):
                    e.set_estimator(mode if mode in ("median", "robust") else "mean")
                    e.set_ci(mode == "ci")
                    e.set_detailed(mode == "detailed")
                    tri, _ = e.triangle(screen=80.0, min_af=15.0)
                    out = [tri] + ([e.last_edge_ci() if mode == "ci" else e.last_edge_detail()] if mode in ("ci", "detailed") else [])
                    for nmax in (0, 1):
                        e.set_max_results(nmax)
                        rect, _ = e.rect(refs, queries, screen=80.0, min_af=15.0)
                        out.append(rect)
                    e.set_max_results(0)
                    res.append(out)
                assert len(res[0][0]) > 5, (m, mode)
                for x, y in zip(*res):
                    assert _bits(x) == _bits(y), (m, mode)
            # search: the query file's records against a database of records
            for e in (ea, eb):
                e.set_estimator("mean")
                e.set_ci(False)
                e.set_detailed(True)
            qp = engine.pack_fasta_many([paths["e.fa"], paths["a.fa"]], threads=2)
            ga, _ = ea.search(qp, per_sequence=True)
            da, sa = ea.last_edge_detail(), ea.last_query_contig_stats
            gb, _ = eb.search([engine.pack_contigs([r]) for r in _records_of([paths["e.fa"], paths["a.fa"]])])
            db_, sb = eb.last_edge_detail(), eb.last_query_contig_stats
            assert len(ga) > 3 and _bits(ga) == _bits(gb) and _bits(da) == _bits(db_)
            assert all(np.array_equal(x, y) for x, y in zip(sa, sb)) and sa[0].tolist() == [1] * 6
            assert ea.n_genomes == n


@pytest.mark.gpu
def test_shim_equals_cpu_reference(built_lib, tmp_path):
    from skder_b200 import daemon

    paths, _ = multi_fastas(tmp_path)
    P = [paths[k] for k in ("a.fa", "b.fa.gz", "c.fa", "d.fa", "e.fa")]

    def both(argv, env=None):
        out, ref = tmp_path / "gpu.tsv", tmp_path / "cpu.tsv"
        for f in (out, ref):
            if f.exists():
                f.unlink()
        assert _run(SHIM, argv + ["-o", str(out)], env) == 0, argv
        assert _run(CPU, argv + ["-o", str(ref)]) == 0, argv
        assert out.read_text() == ref.read_text(), argv
        assert len(out.read_text().splitlines()) > 2, argv
        return out.read_text()

    lst = _lst(tmp_path / "l.txt", P)
    for extra in ([], ["--ci"], ["--detailed"], ["--median"], ["-m", "200"]):
        both(["triangle", "-l", lst, "-E", "-i", "-t", "4"] + extra)
    rl, ql = _lst(tmp_path / "rl.txt", [P[0], P[2], P[4]]), _lst(tmp_path / "ql.txt", [P[1], P[0], P[3]])
    for flags in (["--qi"], ["--ri"], ["--qi", "--ri"]):
        for extra in ([], ["-n", "1"], ["-n", "2", "--detailed"]):
            both(["dist", "--rl", rl, "--ql", ql] + flags + extra)
    db = tmp_path / "db"
    assert _run(SHIM, ["sketch", "-l", _lst(tmp_path / "s.txt", [P[0], P[1], P[2]]), "-o", str(db), "-i"]) == 0
    man = json.load(open(db / "manifest.json"))
    assert man["paths"] == [P[0]] * 3 + [P[1]] * 3 + [P[2]] and man["names"][3:5] == ["dup", "dup"]
    q2 = _lst(tmp_path / "q2.txt", [P[0]])
    for env in ({"SKB_NO_DAEMON": "1"}, {"SKB_DAEMON_IDLE": "120"}):
        try:
            for extra in ([], ["-n", "1"], ["--detailed", "-n", "2"]):
                both(["search", P[4], "-d", str(db), "--ql", q2, "--qi"] + extra, env)
            both(["search", P[4], "-d", str(db)], env)  # whole-file query against a database of records
        finally:
            daemon.stop_for(str(db))
