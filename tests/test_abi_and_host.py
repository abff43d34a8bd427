"""CPU tests of the boundary: the C-ABI library loads and exports every symbol include/skani_b200.h declares,
the host packer agrees with the oracle's ingest, the `skani` shim parses exactly skDER's spellings and fails
loudly (no output file) when it cannot compute.  No compute call is made: there is no GPU here."""
import ctypes as C
import gzip
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported(built_lib):
    from skder_b200 import _lib

    hdr = open(os.path.join(ROOT, "include", "skani_b200.h")).read()
    declared = set(re.findall(r"\b(skb_[a-z0-9_]+)\s*\(", hdr))
    types = {"skb_ctx", "skb_params", "skb_packed", "skb_edge", "skb_pair_detail", "skb_stats", "skb_sketch_view"}
    declared -= types
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    L = C.CDLL(built_lib)
    for name in declared:
        assert hasattr(L, name), name
    # structure layouts the Python side mirrors
    assert C.sizeof(_lib.Edge) == 32 and C.sizeof(_lib.PairDetail) == 80 and C.sizeof(_lib.Stats) == 72


def test_no_cpu_fallback_when_gpu_missing(built_lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from skder_b200 import engine

    with pytest.raises(engine.SkbError, match="no CUDA device|no CPU path"):
        engine.Engine(0)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "skder_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert not re.search(r"#\s*include[^\n]*oracle", src), f  # comments may cite it, code may not use it
                assert "libskani_oracle" not in src and "oracle/_" not in src, f


def test_packer_matches_oracle_ingest(oracle, genomes7, built_lib, tmp_path):
    from skder_b200 import engine

    for f in genomes7[:3]:
        p, s = engine.pack_fasta(f), oracle.Sketch.from_file(f)
        assert (p.n_bases, p.n_contigs, p.first_name) == (s.total_len, s.n_contigs, s.first_name)
        assert np.array_equal(p.contig_lens(), s.contig_lens())
        assert p.n_words % 2 == 0 and p.n_words * 32 >= p.n_bases
    # plain text, CRLF, lowercase, N's, short record dropped, blank lines, junk before the first header
    txt = b"junk\n>c1 first kept\r\nACGTNNacgt" + b"ACGT" * 200 + b"\r\n\r\n>tiny\nACGT\n>c3\n" + b"G" * 600 + b"\n"
    plain = tmp_path / "x.fa"
    plain.write_bytes(txt)
    gz = tmp_path / "x.fa.gz"
    with gzip.open(gz, "wb") as g:
        g.write(txt)
    for path in (plain, gz):
        p, s = engine.pack_fasta(str(path)), oracle.Sketch.from_file(str(path))
        assert p.n_contigs == s.n_contigs == 2 and p.n_bases == s.total_len == 810 + 600
        assert p.first_name == s.first_name == "c1 first kept"
        assert p.total_bases_all == 810 + 4 + 600
    pk = engine.pack_fasta(str(plain))  # keep the owner alive: words() is a view
    w = pk.words()
    codes = [(int(w[j // 32]) >> (2 * (j % 32))) & 3 for j in range(10)]
    assert codes == [0, 1, 2, 3, 0, 0, 0, 1, 2, 3]  # ACGT NN(->A) acgt
    with pytest.raises(engine.SkbError):
        engine.pack_fasta(str(tmp_path / "missing.fa"))
    e = engine.pack_contigs([])
    assert e.n_bases == 0 and e.n_contigs == 0 and e.n_words == 2


def test_cli_parses_exactly_skders_spellings():
    from skder_b200 import cli

    sub, o = cli.parse_args("triangle -l L.txt --min-af 50.0 -E -s 89.5 -t 4 -o out.tsv".split())
    assert sub == "triangle" and (o["list"], o["min_af"], o["screen"], o["threads"], o["out"]) == ("L.txt", 50.0, 89.5, 4, "out.tsv")
    sub, o = cli.parse_args("sketch -l L.txt -o db -t 8".split())
    assert sub == "sketch" and o["out"] == "db"
    sub, o = cli.parse_args("search q.fa -d db -o r.tsv -t 2".split())
    assert sub == "search" and o["positional"] == ["q.fa"] and o["screen"] == 80.0 and o["min_af"] == 15.0
    sub, o = cli.parse_args("dist --rl R --ql Q -s 85 -o Skani_Dist_Output.txt".split())
    assert sub == "dist" and o["screen"] == 85.0
    sub, o = cli.parse_args(["dist", "--rl", "R", "--ql", "Q", "", "-t", "3", "-o", "x"])  # empty -p splice
    assert o["threads"] == 3
    for bad in ("triangle -l L -o o", "triangle -l L -E -o o --fast", "triangle -l L -E -o o -c 30", "dist --rl R -o o",
                "search -d db -o o", "frobnicate", "triangle -l L -E -o o --no-learned-ani", "triangle -l L -E -o o -s x"):
        with pytest.raises(cli.UsageError):
            cli.parse_args(bad.split())


def test_cli_rows_and_loud_failure(tmp_path):
    from skder_b200 import cli
    from skder_b200.engine import EDGE_DTYPE

    e = np.zeros(2, EDGE_DTYPE)
    e[0] = (0, 2, 98.785, 95.456, 92.934)
    e[1] = (1, 2, 100.0, 99.995, 50.0)
    rows = cli.triangle_rows(["/a", "/b", "/c"], ["na", "nb", "nc"], e)
    assert rows[0] == "/a\t/c\t98.78\t95.46\t92.93\tna\tnc\n" or rows[0] == "/a\t/c\t98.79\t95.46\t92.93\tna\tnc\n"
    assert rows[1].split("\t")[2:5] == ["100.00", "100.00" if "%.2f" % 99.995 == "100.00" else "99.99", "50.00"]
    r = cli.rect_rows(["/r1", "/r2", "/q"], ["n1", "n2", "nq"], np.array([(0, 2, 97.0, 80.0, 81.0), (1, 2, 99.0, 90.0, 91.0)], EDGE_DTYPE))
    assert [x.split("\t")[0] for x in r] == ["/r2", "/r1"]  # grouped by query, ANI descending
    assert cli.HEADER == open(os.path.join(ROOT, "tests", "golden", "skder_results", "Skani_Triangle_Edge_Output.txt")).readline()
    # unsupported flag or missing GPU: non-zero exit, NO output file (skDER's runCmd checks only that), a log beside it
    lst = tmp_path / "l.txt"
    lst.write_text("/nonexistent/genome.fa\n")
    out = tmp_path / "edges.tsv"
    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    for argv in (["triangle", "-l", str(lst), "-E", "--slow", "-o", str(out)], ["triangle", "-l", str(lst), "-E", "-o", str(out)]):
        rc = subprocess.call([sys.executable, shim] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        assert rc != 0 and not out.exists()
    assert os.path.exists(str(out) + ".skani_b200.log")


def test_synthetic_generator_is_deterministic():
    from skder_b200 import synth

    a = synth.one_clade(3, 2, 60_000, 11)
    b = synth.one_clade(3, 2, 60_000, 11)
    assert a == b and a != synth.one_clade(4, 2, 60_000, 11)
    g = list(synth.config_genomes("tiny"))
    assert len(g) == 12 and all(sum(map(len, c)) > 20_000 for _, _, c in g)


def _reference_pack(txt, min_len):
    """Plain-Python statement of the packer's rules (csrc/fasta_pack.cpp): '>' starts a record only as the first byte
    of a line, blanks (CR, space, tab) inside sequence lines are dropped, C/G/T in either case are 1/2/3 and every other
    byte is A, records shorter than min_len are left out, text before the first header is ignored."""
    code = {ord("C"): 1, ord("c"): 1, ord("G"): 2, ord("g"): 2, ord("T"): 3, ord("t"): 3}
    recs, cur = [], None
    for line in txt.split(b"\n"):
        if line[:1] == b">":
            cur = []
            recs.append(cur)
        elif cur is not None:
            cur.extend(code.get(c, 0) for c in line if c not in b"\r \t")
    kept = [r for r in recs if len(r) >= min_len and len(r) > 0]
    return [c for r in kept for c in r], [len(r) for r in kept], sum(len(r) for r in recs)


def test_packer_line_shapes_against_plain_python(built_lib, tmp_path):
    """Every line shape the fast paths see: lengths around the 32-base word, pieces that start at any offset inside a
    word, blanks inside lines (slow path), CRLF, IUPAC codes, '>' inside a line, empty lines, no final newline, one
    very long line, records that are rolled back -- plain and gzip, against a plain-Python restatement."""
    from skder_b200 import engine

    rng = np.random.default_rng(5)
    alphabet = np.frombuffer(b"ACGTacgtNnRYKMSWryBDHV>", np.uint8)
    parts = [b"text before any header\nACGT\n"]
    for rec in range(40):
        parts.append(b">rec%d some description\r\n" % rec if rec % 3 == 0 else b">rec%d\n" % rec)
        for _ in range(int(rng.integers(0, 12))):
            n = int(rng.choice([0, 1, 5, 31, 32, 33, 63, 64, 65, 80, 100, 257]))
            line = alphabet[rng.integers(0, len(alphabet), n)].tobytes()
            if line[:1] == b">":
                line = b"A" + line[1:]
            if rng.random() < 0.2 and n > 4:  # blanks inside the line
                k = int(rng.integers(1, n - 1))
                line = line[:k] + rng.choice([b" ", b"\t", b"\r", b"  \t"]) + line[k:]
            parts.append(line + (b"\r\n" if rng.random() < 0.3 else b"\n"))
    parts.append(b">long\n" + alphabet[rng.integers(0, 8, 70_001)].tobytes() + b"\n>last_no_newline\n" + b"ACGT" * 40)
    txt = b"".join(parts)
    plain = tmp_path / "shapes.fa"
    plain.write_bytes(txt)
    gz = tmp_path / "shapes.fa.gz"
    with gzip.open(gz, "wb") as g:
        g.write(txt)
    for min_len in (1, 100, 500):
        codes, lens, total_all = _reference_pack(txt, min_len)
        for path in (plain, gz):
            pk = engine.pack_fasta(str(path), min_len)
            assert (pk.n_bases, pk.n_contigs, pk.total_bases_all) == (len(codes), len(lens), total_all)
            assert pk.contig_lens().tolist() == lens
            w = pk.words()
            got = ((w[:, None] >> (2 * np.arange(32, dtype=np.uint64))[None, :]) & np.uint64(3)).reshape(-1)[: len(codes)]
            assert np.array_equal(got.astype(np.int64), np.array(codes, np.int64))
            assert not np.any(w[(len(codes) + 31) // 32:])  # padding words are zero
            if len(codes) % 32:
                assert int(w[len(codes) // 32]) >> (2 * (len(codes) % 32)) == 0  # and so are the unused bits


def test_bench_host_helpers_without_a_gpu():
    """Host-side pieces of bench.py / multi.py that must not need a device: the clock sampler degrades to
    "unsampled" instead of raising, the NUMA binding says None where sysfs or the GPU is missing, and the checksum of
    a representative set does not depend on the order the loop found them in."""
    sys.path.insert(0, ROOT)
    import bench
    import torch

    from skder_b200 import multi

    assert bench.ids_sha256([5, 1, 9]) == bench.ids_sha256([9, 5, 1]) != bench.ids_sha256([5, 1])
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    assert multi.bind_to_gpu_numa_node(torch, 0) is None
    with bench.ClockSampler(0) as clk:
        pass
    s = clk.summary()
    assert s["sm_mhz"] is None and s["reasons"] == ["unsampled"]


def test_speculative_search_loop_is_the_sequential_loop():
    """bench.py's config4 loop searches the next K unaccounted candidates in one call and applies the results in N50
    order, skipping a candidate an earlier one of its batch accounted for (reference loop: src/skDER/skder.py:116-133).
    Model of that control flow on random hit sets: the representatives equal the one-by-one loop's for every K."""
    rng = np.random.default_rng(7)
    n = 300
    clade = rng.integers(0, 40, n)
    # hits of a query: a random subset of its clade (state-independent, like a search result)
    hits = [np.flatnonzero((clade == clade[g]) & (rng.random(n) < 0.6)) for g in range(n)]
    order = rng.permutation(n).tolist()

    def sequential():
        acc, reps = np.zeros(n, bool), []
        for g in order:
            if acc[g]:
                continue
            reps.append(g)
            acc[hits[g]] = True
            acc[g] = True
        return reps

    def batched(kmax):
        acc, reps, k, pos = np.zeros(n, bool), [], 1, 0
        while pos < n:
            batch, p = [], pos
            while p < n and len(batch) < k:
                if not acc[order[p]]:
                    batch.append(order[p])
                p += 1
            pos = p
            wasted = 0
            for g in batch:
                if acc[g]:
                    wasted += 1
                    continue
                reps.append(g)
                acc[hits[g]] = True
                acc[g] = True
            k = max(1, k // 2) if wasted else min(kmax, k * 2)
        return reps

    want = sequential()
    for kmax in (1, 2, 7, 64):
        assert batched(kmax) == want


def test_search_through_a_running_daemon_loads_neither_numpy_nor_the_engine(tmp_path):
    """skDER's low_mem_greedy loop launches one `skani search` process per representative (reference
    src/skDER/skder.py:116-120).  When the database's daemon answers, the client process must stay light: no numpy,
    no libskani_b200.so.  A stand-in server speaks the daemon's protocol (authenticated Unix socket, JSON bytes)."""
    import json
    import shutil
    import tempfile
    import threading
    from multiprocessing.connection import Listener

    from skder_b200 import daemon

    db = tmp_path / "skani_sketch_all.db"
    db.mkdir()
    # a Unix socket path holds at most 107 bytes, and pytest's tmp_path can be longer: the sockets go to a short
    # private directory instead
    run_dir = tempfile.mkdtemp(prefix="skb-", dir="/tmp")
    env = dict(os.environ, SKB_DAEMON_DIR=run_dir, SKB_DEVICE="0", PYTHONPATH=ROOT)
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

    def serve():
        with Listener(sock, family="AF_UNIX", authkey=key) as ls:
            with ls.accept() as conn:
                msg = json.loads(conn.recv_bytes().decode())
                seen.append(msg)
                with open(msg["out"], "w") as f:
                    f.write("header\n")
                conn.send_bytes(json.dumps({"ok": True}).encode())

    th = threading.Thread(target=serve, daemon=True)
    th.start()
    for _ in range(200):
        if os.path.exists(sock):
            break
        import time

        time.sleep(0.01)
    out = tmp_path / "current_search_results.tsv"
    code = ("import sys; from skder_b200.cli import main; rc = main(sys.argv[1:]); "
            "print('numpy' in sys.modules, 'skder_b200.engine' in sys.modules, rc)")
    try:
        r = subprocess.run([sys.executable, "-c", code, "search", "query.fa", "-d", str(db), "-o", str(out), "-t", "4"],
                           capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=60)
        th.join(timeout=10)
    finally:
        shutil.rmtree(run_dir, ignore_errors=True)
    assert r.stdout.split() == ["False", "False", "0"], r.stdout + r.stderr
    assert out.read_text() == "header\n"
    assert seen and seen[0]["op"] == "search" and seen[0]["query"] == str(tmp_path / "query.fa") and seen[0]["label"] == "query.fa"
    assert "NOT the skani binary" in (tmp_path / "current_search_results.tsv.skani_b200.log").read_text()
