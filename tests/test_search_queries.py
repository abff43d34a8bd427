"""Several queries per `skani search` and skani's -n on search and dist (DESIGN.md section 3): the shim's parser, the
CPU reference (tests/search_queries_ref.py) against an independent restatement, the daemon protocol with a stand-in
server, and on the device: skb_rect's per-query cut against the unrestricted call sorted and cut on the host, the
--ci / --detailed records following their edges, multi-query Engine.search against single searches, the context state,
and the shim end to end against the CPU reference."""
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

SEED = 20261022


def genomes():
    """three clades of five 60 kb genomes, 0.5-5 % apart: every within-clade pair passes the screen at m = 1000"""
    from skder_b200 import synth

    return [g for c in range(3) for g in synth.one_clade(c, 5, 60_000, SEED, d_lo=0.005, d_hi=0.05, max_contigs=3)]


def write_genomes(tmp_path):
    from skder_b200 import synth

    d = tmp_path / "g"
    d.mkdir(exist_ok=True)
    paths = []
    for i, g in enumerate(genomes()):
        p = str(d / ("g%02d.fasta" % i))
        synth.write_fasta(p, g, name="g%02d" % i)
        paths.append(p)
    return paths


def _run(script, argv, env=None, cwd=None):
    return subprocess.call([sys.executable, script] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **(env or {})), cwd=cwd)


# ---- the parser ---------------------------------------------------------------------------------------------------------
def test_parser_queries_and_n(tmp_path):
    from skder_b200 import cli

    ql = tmp_path / "ql.txt"
    ql.write_text("b.fa\nc.fa\n\na.fa\n")
    sub, opt = cli.parse_args(["search", "a.fa", "b.fa", "-d", "db", "-o", "o"])
    assert opt["positional"] == ["a.fa", "b.fa"] and opt["max_results"] == 0
    assert cli.search_queries(opt) == ["a.fa", "b.fa"]
    _, opt = cli.parse_args(["search", "-d", "db", "--ql", str(ql), "-o", "o"])
    assert cli.search_queries(opt) == ["b.fa", "c.fa", "a.fa"]
    _, opt = cli.parse_args(["search", "c.fa", "-d", "db", "--ql", str(ql), "-o", "o", "-n", "2"])
    assert cli.search_queries(opt) == ["c.fa", "b.fa", "a.fa"] and opt["max_results"] == 2
    _, opt = cli.parse_args(["search", "a.fa", "a.fa", "-d", "db", "-o", "o"])
    assert cli.search_queries(opt) == ["a.fa"]
    empty = tmp_path / "empty.txt"
    empty.write_text("\n")
    _, opt = cli.parse_args(["search", "-d", "db", "--ql", str(empty), "-o", "o"])
    with pytest.raises(cli.UsageError):
        cli.search_queries(opt)
    _, opt = cli.parse_args(["dist", "--rl", "r", "--ql", "q", "-o", "o", "-n", "1"])
    assert opt["max_results"] == 1
    _, opt = cli.parse_args(["dist", "--rl", "r", "--ql", "q", "-o", "o", "-n", "007"])
    assert opt["max_results"] == 7
    for argv in (["search", "-d", "db", "-o", "o"],
                 ["triangle", "-l", "l", "-E", "-o", "o", "-n", "1"],
                 ["sketch", "-l", "l", "-o", "o", "-n", "1"],
                 ["dist", "--rl", "r", "--ql", "q", "-o", "o", "-n"],
                 ["dist", "--rl", "r", "--ql", "q", "-o", "o", "-n", "0"],
                 ["dist", "--rl", "r", "--ql", "q", "-o", "o", "-n", "-1"],
                 ["search", "a.fa", "-d", "db", "-o", "o", "-n", "1.5"],
                 ["search", "a.fa", "-d", "db", "-o", "o", "-n", "x"],
                 ["dist", "--rl", "r", "--ql", "q", "-o", "o", "a.fa"]):
        with pytest.raises(cli.UsageError):
            cli.parse_args(argv)


# ---- the CPU reference against a restatement ----------------------------------------------------------------------------
def _restated(rows_by_query, ref_ids, n):
    """per query, the rows sorted by (unrounded oracle ANI descending, reference id) with numpy and cut to n, in their
    first order"""
    from oracle import oracle as O

    sk, out = {}, []
    for rows in rows_by_query:
        for t in rows:
            for p in t[:2]:
                sk.setdefault(p, O.Sketch.from_file(p))
        ani = np.array([O.pair(sk[t[0]], sk[t[1]]).ani for t in rows])
        rid = np.array([ref_ids[t[0]] for t in rows])
        order = np.lexsort((rid, -ani))
        out += [rows[i] for i in np.sort(order[:n])]
    return out


def _rows(path):
    return [ln.split("\t") for ln in open(path).read().splitlines()[1:]]


def test_cpu_reference_against_restatement(oracle, tmp_path):
    paths = write_genomes(tmp_path)
    db_paths = paths[:12]
    lst = tmp_path / "db.txt"
    lst.write_text("".join(p + "\n" for p in db_paths))
    db = tmp_path / "db"
    cpu = os.path.join(ROOT, "tests", "search_queries_ref.py")
    assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"), ["sketch", "-l", str(lst), "-o", str(db)]) == 0
    queries = [paths[1], paths[13], paths[7]]
    ql = tmp_path / "ql.txt"
    ql.write_text("".join(q + "\n" for q in queries[1:] + [queries[0]]))
    single = []
    for q in queries:
        out = tmp_path / "single.tsv"
        assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"), ["search", q, "-d", str(db), "-o", str(out)]) == 0
        single.append(_rows(out))
    assert min(len(r) for r in single) >= 2 and max(len(r) for r in single) >= 4
    ids = {p: i for i, p in enumerate(db_paths)}
    for n in (None, 1, 2, 100):
        out = tmp_path / "multi.tsv"
        extra = ["-n", str(n)] if n else []
        assert _run(cpu, ["search", queries[0], "-d", str(db), "--ql", str(ql), "-o", str(out)] + extra) == 0
        got = _rows(out)
        assert got == (_restated(single, ids, n) if n else [t for r in single for t in r]), n
        if n == 1:
            assert [t[1] for t in got] == queries
    # dist: the same cut on one output
    rl, dq = tmp_path / "rl.txt", tmp_path / "dq.txt"
    rl.write_text("".join(p + "\n" for p in paths[::2]))
    dq.write_text("".join(p + "\n" for p in paths[1::2]))
    full = tmp_path / "full.tsv"
    assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"), ["dist", "--rl", str(rl), "--ql", str(dq), "-o", str(full)]) == 0
    full_rows = _rows(full)
    by_q = {}
    for t in full_rows:
        by_q.setdefault(t[1], []).append(t)
    assert max(len(v) for v in by_q.values()) >= 3
    dist_ids = {p: i for i, p in enumerate(dict.fromkeys(paths[::2] + paths[1::2]))}
    for n in (1, 2):
        out = tmp_path / "dist.tsv"
        assert _run(cpu, ["dist", "--rl", str(rl), "--ql", str(dq), "-o", str(out), "-n", str(n)]) == 0
        assert _rows(out) == _restated(list(by_q.values()), dist_ids, n), n


# ---- the daemon protocol ------------------------------------------------------------------------------------------------
def test_daemon_request_forms():
    from skder_b200 import daemon

    assert daemon.search_queries({"query": "/a.fa", "label": "a.fa"}) == (["/a.fa"], ["a.fa"])
    assert daemon.search_queries({"query": "/a.fa"}) == (["/a.fa"], ["/a.fa"])
    assert daemon.search_queries({"queries": ["/a", "/b"], "labels": ["a", "b"]}) == (["/a", "/b"], ["a", "b"])
    for bad in ({"queries": []}, {"queries": ["/a", "/b"], "labels": ["a"]}):
        with pytest.raises(ValueError):
            daemon.search_queries(bad)


def _shim_through_stand_in(tmp_path, args):
    """the shim's search against a stand-in server; returns the message it sent"""
    from multiprocessing.connection import Listener

    from skder_b200 import daemon

    db = tmp_path / "db"
    db.mkdir(exist_ok=True)
    run_dir = tempfile.mkdtemp(prefix="skb-", dir="/tmp")  # a Unix socket path holds at most 107 bytes
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
        time.sleep(0.01)
    out = tmp_path / "out.tsv"
    try:
        r = subprocess.run([sys.executable, "-m", "skder_b200.cli", "search"] + args + ["-d", str(db), "-o", str(out)],
                           capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=60)
        th.join(timeout=10)
    finally:
        shutil.rmtree(run_dir, ignore_errors=True)
    assert r.returncode == 0, r.stderr
    assert out.read_text() == "header\n"
    return seen[0]


def test_shim_sends_one_or_several_queries(tmp_path):
    msg = _shim_through_stand_in(tmp_path, ["q1.fa"])
    assert msg["query"] == str(tmp_path / "q1.fa") and msg["label"] == "q1.fa"
    assert "queries" not in msg and "max_results" not in msg
    (tmp_path / "ql.txt").write_text("q3.fa\nq1.fa\n")
    msg = _shim_through_stand_in(tmp_path, ["q1.fa", "q2.fa", "--ql", "ql.txt", "-n", "3"])
    assert msg["labels"] == ["q1.fa", "q2.fa", "q3.fa"]
    assert msg["queries"] == [str(tmp_path / q) for q in msg["labels"]]
    assert msg["max_results"] == 3 and "query" not in msg
    log = (tmp_path / "out.tsv.skani_b200.log").read_text()
    assert "-n 3" in log


# ---- on the device ------------------------------------------------------------------------------------------------------
def _bits(a):
    """the bytes of every field (a structured array's padding bytes are not copied by numpy, so its tobytes() is not
    comparable)"""
    if a.dtype.names is None:
        return np.ascontiguousarray(a).tobytes()
    return b"".join(np.ascontiguousarray(a[k]).tobytes() for k in a.dtype.names)


def _cut_on_host(edges, n):
    """indices of the edges skb_rect with -n n keeps: sorted by (query, ANI desc, ref), the first n of each query, back
    in edge order"""
    order = np.lexsort((edges["a"], -edges["ani"], edges["b"]))
    b = edges["b"][order]
    rank = np.arange(len(order)) - np.searchsorted(b, b, side="left")
    return np.sort(order[rank < n]) if n else np.arange(len(edges))


def _dup_set():
    """the clades plus exact copies of three genomes: a query's hits on a genome and its copy tie exactly"""
    g = genomes()
    return g + [g[0], g[5], g[6]]


@pytest.mark.gpu
def test_rect_cut_equals_sorted_and_cut_unrestricted(built_lib):
    from skder_b200 import engine

    contigs = _dup_set()
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(c) for c in contigs])
        e.index()
        refs = [0, 2, 3, 4, 5, 7, 8, 9, 10, 12, 15, 16, 17]
        queries = [1, 6, 11, 13, 14]
        full, _ = e.rect(refs, queries, screen=80.0, min_af=15.0)
        per_q = np.bincount(full["b"])
        assert per_q[queries].min() >= 2
        key = list(zip(full["b"].tolist(), full["ani"].tolist()))
        assert len(set(key)) < len(key)  # exact ties within a query, resolved by reference id
        for n in (1, 2, 3, int(per_q.max()) + 1, 0):
            e.set_max_results(n)
            got, st = e.rect(refs, queries, screen=80.0, min_af=15.0)
            keep = _cut_on_host(full, n)
            assert got.tobytes() == full[keep].tobytes(), n
            assert st.n_edges == len(keep) and e.device_edges()[1] == len(keep)
            want = e.greedy_summary(got, e.n_genomes, 95.0, 15.0)
            have = e.greedy_summary(None, e.n_genomes, 95.0, 15.0)
            assert all(np.array_equal(x, y) for x, y in zip(want, have))
        e.set_max_results(0)


@pytest.mark.gpu
def test_ci_detail_and_estimators_follow_the_kept_edges(built_lib):
    from skder_b200 import engine
    from test_ani_estimators import mag_queries

    mag = mag_queries()
    sets = [("clades", _dup_set(), [0, 2, 3, 4, 5, 7, 8, 9, 10, 12, 15, 16, 17], [1, 6, 11, 13, 14]),
            # the warp, shared-memory CTA and global-scratch finalize routes; genome 4 is a copy of reference 0
            ("routes", mag + [mag[0]], [0, 3, 4], [1, 2])]
    for name, contigs, refs, queries in sets:
        with engine.Engine(0) as e:
            e.add([engine.pack_contigs(c) for c in contigs])
            e.index()
            for mode in ("ci", "detailed", "median", "robust"):
                if mode in ("median", "robust"):
                    e.set_estimator(mode)
                else:
                    getattr(e, "set_" + mode)(True)
                e.set_max_results(0)
                full, _ = e.rect(refs, queries, screen=0.0, min_af=0.0)
                extra = {"ci": e.last_edge_ci, "detailed": e.last_edge_detail}.get(mode)
                full_x = extra() if extra else None
                for n in (1, 2):
                    e.set_max_results(n)
                    got, _ = e.rect(refs, queries, screen=0.0, min_af=0.0)
                    keep = _cut_on_host(full, n)
                    assert len(keep) < len(full) and got.tobytes() == full[keep].tobytes(), (name, mode, n)
                    if extra:
                        assert _bits(extra()) == _bits(full_x[keep]), (name, mode, n)
                e.set_ci(False)
                e.set_detailed(False)
                e.set_estimator("mean")
                e.set_max_results(0)


@pytest.mark.gpu
def test_multi_query_search_equals_single_searches(built_lib):
    from skder_b200 import engine

    contigs = genomes()
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(c) for c in contigs[:10]])
        e.index()
        n_db = e.n_genomes
        qs = [engine.pack_contigs(contigs[k]) for k in (3, 12, 7, 14)]
        for detailed in (False, True):
            e.set_detailed(detailed)
            singles, stats = [], []
            for q in qs:
                ed, _ = e.search(q)
                singles.append((ed, e.last_edge_detail() if detailed else None))
                stats.append(e.last_query_contig_stats)
            assert e.search(qs[0])[0].tobytes() == e.search([qs[0]])[0].tobytes()
            for n in (0, 1):
                e.set_max_results(n)
                multi, _ = e.search(qs)
                det = e.last_edge_detail() if detailed else None
                assert e.n_genomes == n_db
                for k, (ed, sdet) in enumerate(singles):
                    sel = multi["b"] == n_db + k
                    want = ed[_cut_on_host(ed, n)].copy()
                    want["b"] = n_db + k
                    assert multi[sel].tobytes() == want.tobytes(), (k, n)
                    if detailed:
                        assert _bits(det[sel]) == _bits(sdet[_cut_on_host(ed, n)])
                if detailed:
                    cnt, nx = e.last_query_contig_stats
                    assert cnt.tolist() == [s[0][0] for s in stats]
                    assert nx.tolist() == [s[1][0].tolist() for s in stats]
            e.set_max_results(0)
        e.set_detailed(False)


@pytest.mark.gpu
def test_state_survives_clear_and_triangle_is_unaffected(built_lib):
    from skder_b200 import engine
    from skder_b200._lib import SkbError

    contigs = genomes()
    with engine.Engine(0) as e:
        with pytest.raises(SkbError):
            e.set_max_results(-1)
        e.add([engine.pack_contigs(c) for c in contigs])
        e.index()
        tri0, _ = e.triangle()
        full, _ = e.rect(list(range(0, 15, 2)), list(range(1, 15, 2)))
        l0 = e.launches
        e.rect(list(range(0, 15, 2)), list(range(1, 15, 2)))
        plain_launches = e.launches - l0
        e.set_max_results(1)
        e.clear()
        e.add([engine.pack_contigs(c) for c in contigs])
        e.index()
        tri1, st = e.triangle()
        assert tri1.tobytes() == tri0.tobytes() and st.launches > 0
        l0 = e.launches
        got, _ = e.rect(list(range(0, 15, 2)), list(range(1, 15, 2)))
        assert e.launches - l0 > plain_launches
        assert got.tobytes() == full[_cut_on_host(full, 1)].tobytes()
        assert len(got) == len(set(full["b"].tolist())) < len(full)


# ---- the shim end to end ------------------------------------------------------------------------------------------------
def _no_near_ties(paths, rl, ql):
    """distinct ANI values within 1e-9 of each other would let the GPU and the oracle cut differently"""
    from skder_b200 import engine

    with engine.Engine(0) as e:
        e.add_fasta(paths, threads=4)
        e.index()
        full, _ = e.rect(rl, ql, screen=80.0, min_af=15.0)
    for q in set(full["b"].tolist()):
        a = np.sort(full["ani"][full["b"] == q])
        d = np.diff(a)
        assert not np.any((d > 0) & (d < 1e-9)), q


@pytest.mark.gpu
def test_shim_equals_cpu_reference(built_lib, tmp_path):
    from skder_b200 import daemon

    paths = write_genomes(tmp_path)
    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    cpu = os.path.join(ROOT, "tests", "search_queries_ref.py")
    db_paths = paths[:12]
    _no_near_ties(paths, list(range(12)), list(range(15)))
    _no_near_ties(paths, list(range(0, 15, 2)), list(range(1, 15, 2)))
    lst, rl, dq, ql = (tmp_path / f for f in ("db.txt", "rl.txt", "dq.txt", "ql.txt"))
    lst.write_text("".join(p + "\n" for p in db_paths))
    rl.write_text("".join(p + "\n" for p in paths[::2]))
    dq.write_text("".join(p + "\n" for p in paths[1::2]))
    ql.write_text("".join(p + "\n" for p in (paths[13], paths[4], paths[14])))

    def both(argv, env=None):
        out, ref = tmp_path / "gpu.tsv", tmp_path / "cpu.tsv"
        for f in (out, ref):
            if f.exists():
                f.unlink()
        assert _run(shim, argv + ["-o", str(out)], env) == 0, argv
        assert _run(cpu, argv + ["-o", str(ref)]) == 0, argv
        assert out.read_text() == ref.read_text(), argv
        return out.read_text()

    for extra in ([], ["-n", "1"], ["-n", "2", "--ci"], ["-n", "2", "--detailed"], ["-n", "1", "--median"],
                  ["-n", "3", "-m", "200"]):
        text = both(["dist", "--rl", str(rl), "--ql", str(dq), "-t", "4"] + extra)
        assert len(text.splitlines()) > 1
    dbs = {}
    for m in ("1000", "200"):
        dbs[m] = tmp_path / ("db" + m)
        assert _run(shim, ["sketch", "-l", str(lst), "-o", str(dbs[m]), "-t", "4", "-m", m]) == 0
    shapes = {"one": [paths[3]], "positional": [paths[3], paths[13], paths[9]], "ql": ["--ql", str(ql)],
              "mixed": [paths[14], paths[3], "--ql", str(ql)]}
    for env in ({"SKB_NO_DAEMON": "1"}, {"SKB_DAEMON_IDLE": "120"}):
        try:
            for shape, q in shapes.items():
                for extra in ([], ["-n", "1"], ["-n", "2"]):
                    text = both(["search"] + q + ["-d", str(dbs["1000"]), "-t", "2"] + extra, env)
                    if shape == "mixed" and extra == ["-n", "1"]:
                        assert [ln.split("\t")[1] for ln in text.splitlines()[1:]] == [paths[14], paths[3], paths[13],
                                                                                       paths[4]]
            for extra in (["--ci", "-n", "2"], ["--detailed", "-n", "2"], ["--robust", "-n", "1"], ["--detailed"]):
                both(["search", "--ql", str(ql), paths[3], "-d", str(dbs["1000"])] + extra, env)
            both(["search", "--ql", str(ql), paths[3], "-d", str(dbs["200"]), "-n", "2"], env)
        finally:
            daemon.stop_for(str(dbs["1000"]))
            daemon.stop_for(str(dbs["200"]))
    bad = tmp_path / "bad.tsv"
    for argv in (["search", paths[3], str(tmp_path / "missing.fa"), "-d", str(dbs["1000"])],
                 ["search", paths[3], "-d", str(dbs["1000"]), "-n", "0"],
                 ["triangle", "-l", str(lst), "-E", "-n", "1"]):
        for env in ({"SKB_NO_DAEMON": "1"}, {"SKB_DAEMON_IDLE": "120"}):
            try:
                assert _run(shim, argv + ["-o", str(bad)], env) != 0 and not bad.exists(), argv
            finally:
                daemon.stop_for(str(dbs["1000"]))
