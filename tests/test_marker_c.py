"""skani's -m marker compression (DESIGN.md section 3): a canonical 21-mer is a marker iff its hash is below
UINT64_MAX / m.  The shim's parser; the CPU reference (tests/marker_c_ref.py: the unchanged oracle at marker_c = m)
against an independent numpy restatement of the markers; a clade of small genomes whose pairs the prescreen drops at
m = 1000 and keeps at m = 200; the refusal of ranks that sketched at different m; and on the GPU the markers, shared
counts, prescreen decisions and edges against the reference, the database format, the sharded triangle, the context
state and the shim byte for byte against the CPU skani."""
import gzip
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import marker_c_ref as REF  # noqa: E402

MS = (200, 500, 3000)
# small genomes (5-40 kb, 4 per clade, 1-4 % apart): at m = 1000 they hold 0-6 markers, and 9 within-clade pairs
# share none, so the prescreen drops them; at m = 200 every within-clade pair passes
SMALL_LENGTHS = (5_000, 5_000, 7_000, 10_000, 20_000, 40_000)
SMALL_SEED = 20261021


def small_clades():
    from skder_b200 import synth

    return [g for c, L in enumerate(SMALL_LENGTHS)
            for g in synth.one_clade(c, 4, L, SMALL_SEED, d_lo=0.01, d_hi=0.04, max_contigs=3)]


def same_clade(i, j):
    return i // 4 == j // 4


# ---- the markers, restated in numpy ------------------------------------------------------------------------------------
CODE = np.zeros(256, np.uint64)  # non-ACGT -> A, as the oracle's (and skani's) base table
for _ch, _v in ((b"C", 1), (b"c", 1), (b"G", 2), (b"g", 2), (b"T", 3), (b"t", 3)):
    CODE[_ch[0]] = _v
U = np.uint64


def np_mm_hash64(key):
    """minimap2's invertible mix in its shift-add form, wrapping mod 2^64"""
    key = ~(key + (key << U(21)))
    key = key ^ (key >> U(24))
    key = (key + (key << U(3))) + (key << U(8))
    key = key ^ (key >> U(14))
    key = (key + (key << U(2))) + (key << U(4))
    key = key ^ (key >> U(28))
    return key + (key << U(31))


def canonical_21mers(seq):
    c = CODE[np.frombuffer(seq, np.uint8)]
    n = len(c) - 20
    if n <= 0:
        return np.zeros(0, np.uint64)
    f, r = np.zeros(n, np.uint64), np.zeros(n, np.uint64)
    for j in range(21):  # base j of the window: bits 2 (20 - j) of the forward value, complemented at 2 j of the reverse
        w = c[j:j + n]
        f |= w << U(2 * (20 - j))
        r |= (U(3) - w) << U(2 * j)
    return np.minimum(f, r)


def np_markers(contigs, m, min_contig_len=500):
    cm = [canonical_21mers(s) for s in contigs if len(s) >= min_contig_len]
    cm = np.concatenate(cm) if cm else np.zeros(0, np.uint64)
    return np.unique(cm[np_mm_hash64(cm) < U((2 ** 64 - 1) // m)])


def read_fasta(path):
    seqs, cur = [], None
    with gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb") as f:
        for line in f:
            line = line.strip()
            if line.startswith(b">"):
                cur = []
                seqs.append(cur)
            elif cur is not None:
                cur.append(line)
    return [b"".join(s) for s in seqs]


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_parser_takes_m():
    from skder_b200 import cli

    for argv in ("triangle -l L -E -o o", "dist --rl R --ql Q -o o", "sketch -l L -o db"):
        assert cli.parse_args(argv.split())[1]["marker_c"] == 1000
        assert cli.parse_args((argv + " -m 200").split())[1]["marker_c"] == 200
        assert cli.parse_args(("%s -m 1 %s" % tuple(argv.split(" ", 1))).split())[1]["marker_c"] == 1
        for bad in ("0", "-5", "x", "2.5", "1e3", ""):
            with pytest.raises(cli.UsageError):
                cli.parse_args(argv.split() + ["-m", bad])
        with pytest.raises(cli.UsageError):
            cli.parse_args((argv + " -m").split())
    assert cli.parse_args("search q.fa -d db -o o".split())[1]["marker_c"] == 1000
    for bad in ("search q.fa -d db -o o -m 200", "search q.fa -d db -o o -m 1000"):  # the database decides
        with pytest.raises(cli.UsageError):
            cli.parse_args(bad.split())
    # the other sketch options stay refused
    for bad in ("-c 30", "--fast", "--medium", "--slow", "--small-genomes", "--no-learned-ani"):
        for argv in ("triangle -l L -E -o o", "dist --rl R --ql Q -o o", "sketch -l L -o db"):
            with pytest.raises(cli.UsageError):
                cli.parse_args((argv + " -m 200 " + bad).split())


def test_reference_markers_follow_the_definition(oracle, genomes7):
    O = oracle
    for path in genomes7:
        contigs = read_fasta(path)
        assert np.array_equal(O.Sketch.from_file(path, REF.params(1000)).markers(), O.Sketch.from_file(path).markers())
        for m in MS + (1000,):
            got = O.Sketch.from_file(path, REF.params(m)).markers()
            assert np.array_equal(got, np_markers(contigs, m)), (path, m)
            with REF.marker_c(m):  # what the CPU skani runs under
                assert np.array_equal(O.Sketch.from_file(path).markers(), got)
    counts = {}
    for g in small_clades():
        for m in MS + (1000,):
            got = O.Sketch.from_contigs(g, REF.params(m)).markers()
            assert np.array_equal(got, np_markers(g, m)), m
            counts.setdefault(m, []).append(len(got))
    assert min(counts[1000]) <= 2 and min(counts[200]) >= 10  # the clade is small at m = 1000, not at m = 200
    assert sum(counts[200]) > 4 * sum(counts[1000])


def _cpu_edges(sk, params, pairs=None):
    from oracle import skani_cpu

    return {(a, b): (ani, afa, afb) for a, b, ani, afa, afb in skani_cpu.triangle_edges(sk, 80.0, 15.0, 4, params, pairs)}


def test_small_genomes_recovered_at_m200(oracle):
    O = oracle
    gens = small_clades()
    res = {}
    for m in (1000, 200):
        p = REF.params(m)
        sk = [O.Sketch.from_contigs(g, p) for g in gens]
        res[m] = _cpu_edges(sk, p)
    within = {(i, j) for i, j in itertools.combinations(range(len(gens)), 2) if same_clade(i, j)}
    assert set(res[200]) == within  # every within-clade pair, nothing across clades
    missed = within - set(res[1000])
    assert len(missed) >= 5 and set(res[1000]) < set(res[200])
    for ab, v in res[1000].items():  # m decides which pairs are compared, not what a comparison gives
        assert res[200][ab] == v


def _run(script, argv, env=None):
    return subprocess.call([sys.executable, script] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **(env or {})))


def _write_small(tmp_path):
    from skder_b200 import synth

    d = tmp_path / "small"
    d.mkdir()
    paths = []
    for i, g in enumerate(small_clades()):
        p = str(d / ("s%02d.fasta" % i))
        synth.write_fasta(p, g, name="s%02d" % i)
        paths.append(p)
    return paths


def test_cpu_skani_takes_m(oracle, tmp_path):
    """the CPU `skani` the shim is compared with: at -m 1000 it is tests/oracle_skani.py byte for byte; at -m 200 the
    small clade gains the rows it misses at 1000 and keeps the others as they are; sketch -m records m for search"""
    paths = _write_small(tmp_path)
    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in paths))
    outs = {}
    for name, script, extra in (("plain", "oracle_skani.py", []), ("1000", "marker_c_ref.py", ["-m", "1000"]),
                                ("200", "marker_c_ref.py", ["-m", "200"])):
        outs[name] = tmp_path / ("%s.tsv" % name)
        argv = ["triangle", "-l", str(lst), "-E", "-t", "4", "-o", str(outs[name])] + extra
        assert _run(os.path.join(ROOT, "tests", script), argv) == 0
    assert outs["1000"].read_text() == outs["plain"].read_text()
    rows = {k: set(outs[k].read_text().splitlines()) for k in ("1000", "200")}
    assert rows["1000"] < rows["200"] and len(rows["200"] - rows["1000"]) >= 5
    db, sout = tmp_path / "db", tmp_path / "search.tsv"
    assert _run(os.path.join(ROOT, "tests", "marker_c_ref.py"), ["sketch", "-l", str(lst), "-o", str(db), "-m", "200"]) == 0
    assert REF.db_marker_c(str(db)) == 200
    assert _run(os.path.join(ROOT, "tests", "marker_c_ref.py"), ["search", paths[2], "-d", str(db), "-o", str(sout)]) == 0
    hits = {ln.split("\t")[0] for ln in sout.read_text().splitlines()[1:]}
    assert hits == {paths[i] for i in range(4)}  # its whole clade, itself included; at m = 1000 it has no partner
    assert _run(os.path.join(ROOT, "tests", "marker_c_ref.py"), ["sketch", "-l", str(lst), "-o", str(db)]) == 0
    assert _run(os.path.join(ROOT, "tests", "marker_c_ref.py"), ["search", paths[2], "-d", str(db), "-o", str(sout)]) == 0
    assert {ln.split("\t")[0] for ln in sout.read_text().splitlines()[1:]} == {paths[2]}


def _meta_worker(rank, world, port, mcs, q):
    import torch
    import torch.distributed as dist

    from skder_b200 import multi

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    meta = {"n": 2, "n_seeds": 10, "n_mkeys": 5, "marker_c": mcs[rank], "seed_off": np.array([0, 4, 10], np.uint64),
            "total_len": np.array([7000, 9000], np.uint64), "ctg_off": np.array([0, 1, 2], np.uint32),
            "ctg_len": np.array([7000, 9000], np.uint32)}
    try:
        metas = multi._exchange_meta(meta, dist, torch, None)
        q.put((rank, [m["marker_c"] for m in metas]))
    except ValueError as e:
        q.put((rank, "refused: %s" % e))
    dist.destroy_process_group()


@pytest.mark.parametrize("mcs", [(200, 200), (1000, 200)], ids=["same", "mismatched"])
def test_ranks_must_agree_on_m(mcs):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29300 + os.getpid() % 150 + (150 if mcs[0] != mcs[1] else 0)
    procs = [ctx.Process(target=_meta_worker, args=(r, 2, port, mcs, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    if mcs[0] == mcs[1]:
        assert got == {0: list(mcs), 1: list(mcs)}
    else:  # every rank refuses, so none waits for a collective the others skip
        assert all(v.startswith("refused") and "[1000, 200]" in v for v in got.values())


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _screened(e, screen):
    """the pairs skb_screen_triangle keeps"""
    import torch

    from skder_b200 import multi

    ptr, n, _ = e.screen_triangle(screen)
    v = multi._dev_tensor(torch, ptr, n, torch.device("cuda", e.device)).cpu().numpy().view(np.uint64)
    return {(int(x) >> 32, int(x) & 0xFFFFFFFF) for x in v}


def _edge_map(edges):
    return {(int(x["a"]), int(x["b"])): (float(x["ani"]), float(x["af_a"]), float(x["af_b"])) for x in edges}


def _assert_edges_equal(got, want, what):
    """same pairs; ANI/AF within 1e-12 (percent) with the same 2-decimal text"""
    assert set(got) == set(want), (what, sorted(set(got) ^ set(want))[:5])
    for ab, g in got.items():
        w = want[ab]
        assert all(abs(x - y) <= 1e-12 for x, y in zip(g, w)), (what, ab, g, w)
        assert ["%.2f" % x for x in g] == ["%.2f" % y for y in w], (what, ab)


def _engine(packed, m, index=True):
    from skder_b200 import engine

    e = engine.Engine(0)
    e.set_marker_compression(m)
    e.add(packed)
    if index:
        e.index()
    return e


@pytest.fixture(scope="module")
def sets(built_lib, genomes7, oracle):
    from skder_b200 import engine

    small = small_clades()
    return {"genomes7": (engine.pack_fasta_many(genomes7, threads=4), lambda p: [oracle.Sketch.from_file(f, p) for f in genomes7]),
            "small": ([engine.pack_contigs(g) for g in small], lambda p: [oracle.Sketch.from_contigs(g, p) for g in small])}


@pytest.mark.gpu
@pytest.mark.parametrize("m", MS)
def test_markers_counts_and_screen_bit_exact(sets, oracle, m):
    O = oracle
    p = REF.params(m)
    for name, (packed, sketch) in sets.items():
        sk = sketch(p)
        with _engine(packed, m) as e:
            assert e.marker_compression == m
            for g, s in enumerate(sk):
                assert np.array_equal(e.markers(g), s.markers()), (name, m, g)
                assert np.array_equal(e.seeds(g), s.seeds()), (name, m, g)  # seeds do not depend on m
            pairs = list(itertools.combinations(range(len(sk)), 2))
            got = e.shared_markers([a for a, _ in pairs], [b for _, b in pairs])
            assert list(got) == [O.screen(sk[a], sk[b], 0.8, p)[0] for a, b in pairs], (name, m)
            for screen in (80.0, 89.5):
                want = {(a, b) for a, b in pairs if O.screen(sk[a], sk[b], screen / 100.0, p)[1]}
                assert _screened(e, screen) == want, (name, m, screen)


@pytest.mark.gpu
def test_edges_equal_reference_in_triangle_rect_and_search(sets, oracle):
    O = oracle
    for name, (packed, sketch) in sets.items():
        for m in (200, 1000):
            p = REF.params(m)
            sk = sketch(p)
            n = len(sk)
            want = _cpu_edges(sk, p)
            with _engine(packed, m) as e:
                tri = _edge_map(e.triangle(80.0, 15.0)[0])
                _assert_edges_equal(tri, want, (name, m, "triangle"))
                refs, queries = list(range(0, n, 2)), list(range(1, n, 2))
                rect = _edge_map(e.rect(refs, queries, 80.0, 15.0)[0])
                want_rect = {}
                for b in queries:
                    for a in refs:
                        if O.screen(sk[a], sk[b], 0.8, p)[1]:
                            r = O.pair(sk[a], sk[b], p)
                            if r.ani >= 0 and max(r.af_a, r.af_b) * 100 >= 15.0:
                                want_rect[a, b] = (100 * r.ani, 100 * r.af_a, 100 * r.af_b)
                _assert_edges_equal(rect, want_rect, (name, m, "rect"))
            # search: the database without genome q, q sketched as the query at the database's m
            for q in (2, n - 1):
                db = [packed[i] for i in range(n) if i != q]
                ids = [i for i in range(n) if i != q]
                with _engine(db, m) as e:
                    res = e.search(packed[q], 80.0, 15.0)[0]  # a = database id, b = the query
                got = {(ids[a], q): v for (a, _), v in _edge_map(res).items()}
                want_s = {}
                for a in ids:
                    if O.screen(sk[a], sk[q], 0.8, p)[1]:
                        r = O.pair(sk[a], sk[q], p)
                        if r.ani >= 0 and max(r.af_a, r.af_b) * 100 >= 15.0:
                            want_s[a, q] = (100 * r.ani, 100 * r.af_a, 100 * r.af_b)
                _assert_edges_equal(got, want_s, (name, m, "search", q))
    # the small clade: m = 200 finds the within-clade edges m = 1000 misses, and leaves the others as they were
    packed, _ = sets["small"]
    with _engine(packed, 1000) as e:
        at1000 = _edge_map(e.triangle(80.0, 15.0)[0])
    with _engine(packed, 200) as e:
        at200 = _edge_map(e.triangle(80.0, 15.0)[0])
    assert len(set(at200) - set(at1000)) >= 5 and all(same_clade(a, b) for a, b in at200)
    assert all(at200[ab] == v for ab, v in at1000.items())


@pytest.mark.gpu
def test_db_round_trip(sets, oracle, tmp_path):
    from skder_b200 import engine

    packed, sketch = sets["small"]
    n = len(packed)
    # m = 1000: the SKB200v1 file, as a context that never heard of -m writes it
    for d, m in (("plain", None), ("m1000", 1000), ("m200", 200)):
        with engine.Engine(0) as e:
            if m is not None:
                e.set_marker_compression(m)
            e.add(packed[:-1])
            e.save(str(tmp_path / d))
    v1 = (tmp_path / "plain" / "sketches.skb").read_bytes()
    assert v1[:8] == b"SKB200v1" and (tmp_path / "m1000" / "sketches.skb").read_bytes() == v1
    v2 = (tmp_path / "m200" / "sketches.skb").read_bytes()
    assert v2[:8] == b"SKB200v2" and int.from_bytes(v2[8:16], "little") == 200
    n_mk1 = int.from_bytes(v1[24:32], "little")
    n_mk2 = int.from_bytes(v2[32:40], "little")
    assert n_mk2 > n_mk1 and v2[16:32] == v1[8:24] and v2[40:48] == v1[32:40]  # n, seeds, contigs as v1; more markers
    assert len(v2) == len(v1) + 8 + 8 * (n_mk2 - n_mk1)
    assert REF.db_marker_c(str(tmp_path / "m200")) == 200 and REF.db_marker_c(str(tmp_path / "plain")) == 1000
    for d, m in (("plain", 1000), ("m200", 200)):
        with engine.Engine(0) as e:
            e.set_marker_compression(500)  # the file's m replaces the context's
            e.load(str(tmp_path / d))
            assert e.marker_compression == m
            e.index()
            sk = sketch(REF.params(m))
            for g in range(n - 1):
                assert np.array_equal(e.markers(g), sk[g].markers())
            with _engine(packed[:-1], m) as ref:
                assert e.triangle(80.0, 15.0)[0].tobytes() == ref.triangle(80.0, 15.0)[0].tobytes()
                # the query of a search is sketched at the database's m
                assert e.search(packed[-1], 80.0, 15.0)[0].tobytes() == ref.search(packed[-1], 80.0, 15.0)[0].tobytes()
            e.add([packed[-1]])
            e.index_append()
            assert np.array_equal(e.markers(n - 1), sk[n - 1].markers())
            with pytest.raises(engine.SkbError, match=r"\(-5\)"):  # holds genomes sketched at m
                e.set_marker_compression(m + 1)


@pytest.mark.gpu
def test_sharded_triangle_at_m200(sets):
    packed, _ = sets["small"]
    with _engine(packed, 200) as e:
        want = _edge_map(e.triangle(80.0, 15.0)[0])
    got = {}
    n = len(packed)
    for first, count in [(0, n // 2), (n // 2, n - n // 2)]:
        with _engine(packed, 200) as e2:
            e2.set_owned(first, count)
            e2.index()
            ptr, k, _ = e2.screen_triangle(80.0)
            got.update(_edge_map(e2.pairs_edges(ptr, k, owned_only=True, min_af=15.0)[0]))
    assert got == want


@pytest.mark.gpu
def test_context_state(sets):
    from skder_b200 import engine
    from skder_b200._lib import SkbError

    packed, _ = sets["small"]
    with engine.Engine(0) as fresh:
        l0 = fresh.launches
        fresh.add(packed)
        fresh.index()
        want_edges = fresh.triangle(80.0, 15.0)[0].tobytes()
        want_launches = fresh.launches - l0
        want_markers = [fresh.markers(g) for g in range(len(packed))]
    with engine.Engine(0) as e:
        assert e.marker_compression == 1000
        for bad in (0, -5):
            with pytest.raises(SkbError, match=r"\(-1\)"):
                e.set_marker_compression(bad)
        assert e.marker_compression == 1000
        e.set_marker_compression(200)
        e.add(packed)
        e.set_marker_compression(200)  # the value it has: fine
        with pytest.raises(SkbError, match=r"\(-5\)"):
            e.set_marker_compression(1000)
        e.index()
        at200 = e.triangle(80.0, 15.0)[0].tobytes()
        e.clear()
        assert e.marker_compression == 200  # survives clear
        e.add(packed)
        e.index()
        assert e.triangle(80.0, 15.0)[0].tobytes() == at200
        e.clear()
        e.set_marker_compression(1000)  # and back: exactly what a context that was never changed computes
        l0 = e.launches
        e.add(packed)
        e.index()
        assert e.triangle(80.0, 15.0)[0].tobytes() == want_edges
        assert e.launches - l0 == want_launches
        assert all(np.array_equal(e.markers(g), w) for g, w in enumerate(want_markers))


def _shim_setup(tmp_path, genomes7):
    paths = _write_small(tmp_path) + list(genomes7[:3])
    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in paths))
    rl, ql = tmp_path / "r.txt", tmp_path / "q.txt"
    rl.write_text("".join(p + "\n" for p in paths[0::2]))
    ql.write_text("".join(p + "\n" for p in paths[1::2]))
    return paths, lst, rl, ql


def _both(tmp_path, argv, env=None):
    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    cpu = os.path.join(ROOT, "tests", "marker_c_ref.py")
    out, ref = tmp_path / "gpu.tsv", tmp_path / "cpu.tsv"
    for f in (out, ref):
        if f.exists():
            f.unlink()
    assert _run(shim, argv + ["-o", str(out)], env) == 0, argv
    assert _run(cpu, argv + ["-o", str(ref)]) == 0, argv
    assert out.read_text() == ref.read_text(), argv
    return out


@pytest.mark.gpu
def test_shim_end_to_end_equals_cpu_skani(genomes7, built_lib, tmp_path):
    from skder_b200 import daemon

    paths, lst, rl, ql = _shim_setup(tmp_path, genomes7)
    rows = {}
    for m in ("1000", "200"):
        out = _both(tmp_path, ["triangle", "-l", str(lst), "--min-af", "15.0", "-E", "-t", "4", "-m", m])
        rows[m] = set(out.read_text().splitlines())
        log = open(str(out) + ".skani_b200.log").read()
        assert ("-m 200" in log) == (m == "200")
        _both(tmp_path, ["dist", "--rl", str(rl), "--ql", str(ql), "-m", m])
    assert rows["1000"] < rows["200"]
    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    db = tmp_path / "db"
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(db), "-t", "4", "-m", "200"]) == 0
    assert (db / "sketches.skb").read_bytes()[:8] == b"SKB200v2"
    for q in (paths[2], paths[-1]):
        out = _both(tmp_path, ["search", q, "-d", str(db), "-t", "2"], {"SKB_NO_DAEMON": "1"})
    assert len(out.read_text().splitlines()) > 1
    try:
        for q in (paths[2], paths[5], paths[2]):  # one resident server
            _both(tmp_path, ["search", q, "-d", str(db), "-t", "2"], {"SKB_DAEMON_IDLE": "120"})
        assert daemon.request(str(db), 0, {"op": "ping"}, timeout=5.0)["n"] == len(paths)
    finally:
        daemon.stop_for(str(db))
    bad = tmp_path / "bad.tsv"
    for argv in (["search", paths[2], "-d", str(db), "-m", "200"], ["triangle", "-l", str(lst), "-E", "-m", "0"],
                 ["triangle", "-l", str(lst), "-E", "-m", "200", "-c", "30"]):
        assert _run(shim, argv + ["-o", str(bad)]) != 0 and not bad.exists()


@pytest.mark.gpu
def test_shim_m200_with_estimators_ci_and_detailed(genomes7, built_lib, tmp_path):
    """-m changes which rows there are, not what the --median / --robust / --ci / --detailed columns mean"""
    from skder_b200 import daemon

    paths, lst, rl, ql = _shim_setup(tmp_path, genomes7)
    for extra in (["--median"], ["--robust"], ["--ci"], ["--detailed"]):
        out = _both(tmp_path, ["triangle", "-l", str(lst), "-E", "-t", "4", "-m", "200"] + extra)
        assert len(out.read_text().splitlines()) > 1 + 36  # the small clade alone has 36 edges at m = 200
        _both(tmp_path, ["dist", "--rl", str(rl), "--ql", str(ql), "-m", "200"] + extra)
    db = tmp_path / "db"
    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    assert _run(shim, ["sketch", "-l", str(lst), "-o", str(db), "-t", "4", "-m", "200"]) == 0
    try:
        for extra in (["--ci"], ["--detailed"], ["--median"]):
            _both(tmp_path, ["search", paths[2], "-d", str(db), "-t", "2"] + extra, {"SKB_DAEMON_IDLE": "120"})
    finally:
        daemon.stop_for(str(db))
