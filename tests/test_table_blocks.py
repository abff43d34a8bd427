"""On-demand seed tables (DESIGN.md section 2): with SKB_TABLE_BUDGET_MB below the size of every genome's table, skb_index
switches the context to tables built per edge call in blocks of reference genomes.  Every output must be byte-identical
to the resident run on the same inputs: seeds with their repeat flags, edges, --ci / --detailed records, -n cuts, the
--median / --robust estimators, the greedy summary, the full matrix, skb_pairs_detail, Engine.search, pairs_edges, and
the shim's triangle, dist and search with and without the daemon.  Budgets give one block, several blocks, and one
genome per block; the block count is read back through skb_table_blocks."""
import contextlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 20261022
MIB = float(1 << 20)


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items() if v is not None})
    for k, v in kv.items():
        if v is None:
            os.environ.pop(k, None)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def synthetic_sets():
    """clades; fragmented genomes (up to 200 contigs); repeat-rich genomes with small indels"""
    from skder_b200 import synth

    clades = [g for c in range(3) for g in synth.one_clade(c, 5, 80_000, SEED, d_lo=0.002, d_hi=0.04, max_contigs=4)]
    frag = [g for c in range(2) for g in synth.one_clade(10 + c, 5, 120_000, SEED, d_lo=0.005, d_hi=0.03, max_contigs=200)]
    reps = [g for c in range(2) for g in synth.one_clade(20 + c, 5, 100_000, SEED, d_lo=0.002, d_hi=0.03, max_contigs=8,
                                                         realistic=True)]
    return {"clades": clades, "fragmented": frag, "repeats": reps}


def packed_sets(genomes7):
    from skder_b200 import engine

    sets = {k: [engine.pack_contigs(c) for c in v] for k, v in synthetic_sets().items()}
    sets["genomes7"] = engine.pack_fasta_many(genomes7, 4)
    return sets


def table_bytes(e):
    """the size skb_index weighs against the budget, at SKB_TAB_X2 = 4"""
    seeds = sum(e.sizes(g)["n_seeds"] for g in range(e.n_genomes))
    return (seeds * 2 + e.n_genomes) * 32.0


def budgets(total):
    """one block (the references' tables fit), several blocks, one genome per block"""
    return {"one": 0.95 * total / MIB, "several": 0.2 * total / MIB, "per_genome": 1e-9}


def fields(a):
    """the named fields of a structured array as bytes (a copy need not carry the bytes between them)"""
    return b"".join(a[f].tobytes() for f in a.dtype.names)


def run_battery(packed, tmp, budget_mb):
    """every output of one context over `packed`, as bytes; and the block counts of its edge calls"""
    from skder_b200 import engine

    out, blocks = {}, {}
    with env(SKB_TABLE_BUDGET_MB=budget_mb, SKB_TAB_X2=4), engine.Engine(0) as e:
        e.add(packed)
        e.index()
        n = e.n_genomes
        out["on_demand"] = e.table_blocks()[0]
        out["seeds"] = b"".join(e.seeds(g).tobytes() for g in range(n))

        def call(name, f):
            r = f()
            blocks[name] = e.table_blocks()[1]
            return r

        tri, st = call("triangle", lambda: e.triangle(screen=80.0, min_af=15.0))
        out["triangle"] = tri.tobytes()
        out["stats"] = (st.n_pairs_total, st.n_pairs_screened, st.n_edges, st.sum_query_seeds, st.sum_anchors)
        c, o, m = e.greedy_summary(None, n, 95.0, 15.0)
        out["summary"] = c.tobytes() + o.tobytes() + m.tobytes()
        path = os.path.join(tmp, "matrix.txt")
        e.write_matrix(path, ["g%d" % g for g in range(n)], "ani")
        out["matrix"] = open(path, "rb").read()
        for flag in ("ci", "detailed"):
            getattr(e, "set_" + flag)(True)
            t, _ = call("triangle_" + flag, lambda: e.triangle(screen=80.0, min_af=15.0))
            out["triangle_" + flag] = t.tobytes() + (e.last_edge_ci().tobytes() if flag == "ci" else fields(e.last_edge_detail()))
            getattr(e, "set_" + flag)(False)
        for est in ("median", "robust"):
            e.set_estimator(est)
            t, _ = call("triangle_" + est, lambda: e.triangle(screen=80.0, min_af=15.0))
            out["triangle_" + est] = t.tobytes()
        e.set_estimator("mean")
        refs, queries = list(range(0, n, 2)), list(range(1, n, 2))
        for k in (0, 1, 2):
            e.set_max_results(k)
            e.set_detailed(True)
            r, _ = call("rect_n%d" % k, lambda: e.rect(refs, queries, screen=80.0, min_af=15.0))
            out["rect_n%d" % k] = r.tobytes() + fields(e.last_edge_detail())
            c, o, m = e.greedy_summary(None, n, 95.0, 15.0)
            out["rect_summary_n%d" % k] = c.tobytes() + o.tobytes() + m.tobytes()
            e.set_detailed(False)
        e.set_max_results(0)
        ptr, np_, _ = e.screen_triangle(screen=80.0)
        pe, _ = call("pairs_edges", lambda: e.pairs_edges(ptr, np_, owned_only=False, min_af=15.0))
        out["pairs_edges"] = pe.tobytes()
        rng = np.random.default_rng(SEED)
        a, b = np.triu_indices(n, 1)
        order = rng.permutation(len(a))
        d = call("pairs_detail", lambda: e.pairs_detail(a[order], b[order]))
        out["pairs_detail"] = bytes(memoryview(d))
    with env(SKB_TABLE_BUDGET_MB=budget_mb, SKB_TAB_X2=4), engine.Engine(0) as e:
        # a database of the first genomes, searched by the others: append, search, pop, repeated
        n_db = max(3, len(packed) * 2 // 3)
        e.add(packed[:n_db])
        e.index()
        for rep in range(2):
            for k in (0, 2):
                e.set_max_results(k)
                for q in (packed[n_db:], packed[n_db:n_db + 1], packed[-1:]):
                    r, _ = call("search", lambda: e.search(q, screen=80.0, min_af=15.0))
                    out["search_%d_%d_%d" % (rep, k, len(q))] = r.tobytes()
                    assert e.n_genomes == n_db
        out["db_seeds"] = b"".join(e.seeds(g).tobytes() for g in range(n_db))
    return out, blocks


@pytest.mark.gpu
def test_on_demand_tables_equal_resident(built_lib, genomes7, tmp_path):
    from skder_b200 import engine

    for name, packed in packed_sets(genomes7).items():
        with env(SKB_TAB_X2=4), engine.Engine(0) as e:
            e.add(packed)
            e.index()
            total = table_bytes(e)
        want, wblocks = run_battery(packed, str(tmp_path), None)
        assert want["on_demand"] is False and set(wblocks.values()) == {0}, name
        assert len(want["triangle"]) > 0, name
        for label, mb in budgets(total).items():
            got, blocks = run_battery(packed, str(tmp_path), mb)
            assert got["on_demand"] is True, (name, label)
            for k in want:
                if k != "on_demand":
                    assert got[k] == want[k], (name, label, k)
            if label == "one":
                assert blocks["triangle"] == 1, (name, blocks)
            else:
                assert blocks["triangle"] > 1 and blocks["pairs_detail"] > 1, (name, label, blocks)
            if label == "per_genome":
                # every reference of a surviving pair in a block of its own
                a = np.frombuffer(want["triangle"], dtype=engine.EDGE_DTYPE)
                assert blocks["triangle"] >= len(set(a["a"].tolist()) | set(a["b"].tolist())) // 2, (name, blocks)


@pytest.mark.gpu
def test_resident_tables_when_they_fit(built_lib, genomes7):
    """no cap, or a cap above every table: resident tables, the same launches as without the variable"""
    from skder_b200 import engine

    packed = engine.pack_fasta_many(genomes7, 4)
    launches = []
    for mb in (None, 1e6):
        with env(SKB_TABLE_BUDGET_MB=mb), engine.Engine(0) as e:
            e.add(packed)
            e.index()
            l0 = e.launches
            e.triangle()
            launches.append(e.launches - l0)
            assert e.table_blocks() == (False, 0)
    assert launches[0] == launches[1]


@pytest.mark.gpu
def test_unsorted_pairs_edges_keep_their_order(built_lib):
    """skb_pairs_edges over a caller's unsorted pair list: on-demand blocks return the edges in the list's order, as the
    resident pass does"""
    import torch
    from skder_b200 import engine

    packed = [engine.pack_contigs(c) for c in synthetic_sets()["clades"]]
    a, b = np.triu_indices(len(packed), 1)
    pairs = (a.astype(np.uint64) << np.uint64(32)) | b.astype(np.uint64)
    pairs = pairs[np.random.default_rng(SEED).permutation(len(pairs))]
    dev = torch.from_numpy(pairs.view(np.int64)).cuda()
    torch.cuda.synchronize()
    got = {}
    for label, mb in (("resident", None), ("blocks", 1e-9)):
        with env(SKB_TABLE_BUDGET_MB=mb, SKB_TAB_X2=4), engine.Engine(0) as e:
            e.add(packed)
            e.index()
            e.set_detailed(True)
            edges, _ = e.pairs_edges(dev.data_ptr(), len(pairs), owned_only=False, min_af=15.0)
            got[label] = edges.tobytes() + fields(e.last_edge_detail())
            on, blocks = e.table_blocks()
            assert (on, blocks) == (False, 0) if mb is None else (on and blocks > 1), (label, on, blocks)
            key = edges["a"].astype(np.uint64) << np.uint64(32) | edges["b"].astype(np.uint64)
            assert len(edges) > 2 and np.any(np.diff(key.astype(np.int64)) < 0), label  # not (a, b) order
    assert got["blocks"] == got["resident"]


@pytest.mark.gpu
def test_small_set_stays_resident_on_a_busy_device(built_lib, genomes7):
    """with less free memory than the 40 GiB table_density keeps aside -- another tenant holding the rest -- a small
    set's tables stay resident, as before on-demand tables existed, with the same edges"""
    import torch
    from skder_b200 import engine

    packed = engine.pack_fasta_many(genomes7, 4)

    def run():
        with env(SKB_TABLE_BUDGET_MB=None), engine.Engine(0) as e:
            e.add(packed)
            e.index()
            edges, _ = e.triangle()
            return e.table_blocks(), edges.tobytes()

    want = run()
    free, _ = torch.cuda.mem_get_info(0)
    keep = 24 << 30
    hog = torch.empty(max(0, free - keep), dtype=torch.uint8, device="cuda") if free > keep else None
    try:
        assert torch.cuda.mem_get_info(0)[0] < 40 << 30
        got = run()
    finally:
        del hog
        torch.cuda.empty_cache()
    assert want[0] == (False, 0) and got == want


def _run(argv, extra_env):
    shim = os.path.join(ROOT, "skder_b200", "bin", "skani")
    return subprocess.call([sys.executable, shim] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                           env=dict(os.environ, **extra_env))


@pytest.mark.gpu
def test_shim_on_demand_equals_resident(built_lib, tmp_path):
    from skder_b200 import daemon, synth

    paths = []
    for i, g in enumerate(synthetic_sets()["clades"]):
        p = str(tmp_path / ("g%02d.fasta" % i))
        synth.write_fasta(p, g, name="g%02d" % i)
        paths.append(p)
    lst, rl, ql = (tmp_path / f for f in ("all.txt", "rl.txt", "ql.txt"))
    lst.write_text("".join(p + "\n" for p in paths[:12]))
    rl.write_text("".join(p + "\n" for p in paths[::2]))
    ql.write_text("".join(p + "\n" for p in paths[1::2]))
    db = tmp_path / "db"
    assert _run(["sketch", "-l", str(lst), "-o", str(db)], {"SKB_NO_DAEMON": "1"}) == 0
    commands = {
        "triangle": ["triangle", "-l", str(lst), "-E"],
        "triangle_detailed": ["triangle", "-l", str(lst), "-E", "--detailed"],
        "dist": ["dist", "--rl", str(rl), "--ql", str(ql), "-n", "2", "--ci"],
        "search": ["search", paths[12], paths[13], paths[14], "-d", str(db), "-n", "2"],
        "search_detailed": ["search", paths[14], paths[3], "-d", str(db), "--detailed"],
    }
    outs = {}
    for budget in (None, "1e-9", "0.05"):
        for mode in ({"SKB_NO_DAEMON": "1"}, {"SKB_DAEMON_IDLE": "120"}):
            e = dict(mode, SKB_PHASE_LOG="1", **({"SKB_TABLE_BUDGET_MB": budget} if budget else {}))
            try:
                for name, argv in commands.items():
                    out = tmp_path / "out.tsv"
                    log = tmp_path / "out.tsv.skani_b200.phases.json"
                    for f in (out, log):
                        if f.exists():
                            f.unlink()
                    assert _run(argv + ["-o", str(out)], e) == 0, (name, e)
                    outs.setdefault(name, set()).add(out.read_bytes())
                    # the run really used the tables the budget asks for: the phase log of an in-process run, the
                    # daemon's own report for a search it served
                    if argv[0] == "search" and "SKB_NO_DAEMON" not in mode:
                        tb = daemon.request(str(db), 0, {"op": "ping"})["table_blocks"]
                    else:
                        tb = json.loads(log.read_text())["table_blocks"]
                    assert tb["on_demand"] is (budget is not None), (name, e, tb)
                    assert (tb["blocks"] >= 1) if budget else (tb["blocks"] == 0), (name, e, tb)
            finally:
                daemon.stop_for(str(db))
    for name, texts in outs.items():
        assert len(texts) == 1, name
        assert len(next(iter(texts)).splitlines()) > 1, name
