"""On-demand seed tables (DESIGN.md section 2) on one GPU: what they cost where resident tables fit, and what they hold
where resident tables would not.

  python tools/bench_table_blocks.py [--rounds 3] [--copies 36] [--skip-triangle] [--skip-search] [--skip-capacity]
                                     [--out result.json]

1. config3 triangle (bench.py's default workload and thresholds, -s 89.5 --min-af 50): resident tables against table
   budgets (SKB_TABLE_BUDGET_MB) that force about 2, 4 and 8 blocks, re-indexed per mode on one context and alternated
   over --rounds: device time of skb_triangle (CUDA events on the context's stream), blocks, launches, and the sha256 of
   the edge bytes, which must be one value.
2. A 64-query Engine.search batch against a config4-sized database (the first 19,936 genomes of config4's 20,000; the
   last 64 are the queries), resident against on-demand tables at a budget of an eighth of the tables: device time,
   blocks, and the sha256 of the hits.
3. Capacity: config3's sketches imported --copies times (skb_import_sketches) into a second context.  At 1.1 MB per 5 Mbp
   genome with the densest resident tables (DESIGN.md section 2) such a database would need more than the device holds;
   with on-demand tables it indexes and answers.  64 queries of the original set are searched against it, and each
   query's hits must equal its hits in the original set, repeated once per copy.

Prints one JSON line with the card's name, power limit and max SM clock read in the same run.
"""
import argparse
import contextlib
import hashlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_estimators import card  # noqa: E402

SCREEN, MIN_AF = 89.5, 50.0
MIB = float(1 << 20)


@contextlib.contextmanager
def budget(mb):
    old = os.environ.pop("SKB_TABLE_BUDGET_MB", None)
    if mb is not None:
        os.environ["SKB_TABLE_BUDGET_MB"] = repr(mb)
    try:
        yield
    finally:
        os.environ.pop("SKB_TABLE_BUDGET_MB", None)
        if old is not None:
            os.environ["SKB_TABLE_BUDGET_MB"] = old


def sha(a):
    return hashlib.sha256(a.tobytes()).hexdigest()


def table_bytes(eng, x2):
    """the size skb_index weighs against the budget"""
    seeds = sum(eng.sizes(g)["n_seeds"] for g in range(eng.n_genomes))
    return (seeds * x2 / 2 + eng.n_genomes) * 32.0


def timed(eng, f):
    l0 = eng.launches
    eng.timer_start()
    r = f()
    ms = eng.timer_stop()
    return r, ms, eng.launches - l0


def triangle_modes(eng, rounds):
    total = table_bytes(eng, 4)
    modes = {"resident": None}
    for k in (2, 4, 8):
        modes["blocks%d" % k] = total / k * 1.02 / MIB
    res = {m: {"ms": []} for m in modes}
    for r in range(rounds + 1):  # round 0 warms every mode up
        names = list(modes)
        for m in names[r % len(names):] + names[:r % len(names)]:
            with budget(modes[m]):
                eng.index()
                eng.triangle(SCREEN, MIN_AF)  # steady state: the table buffer and scratch are allocated
                (edges, st), ms, launches = timed(eng, lambda: eng.triangle(SCREEN, MIN_AF))
                on, blocks = eng.table_blocks()
            if r:
                res[m]["ms"].append(round(ms, 1))
            res[m].update(on_demand=on, blocks=blocks, launches=launches, edges=len(edges), edges_sha256=sha(edges),
                          budget_mb=None if modes[m] is None else round(modes[m], 1))
    with budget(None):
        eng.index()
    assert len({v["edges_sha256"] for v in res.values()}) == 1, res
    for v in res.values():
        v["median_ms"] = sorted(v["ms"])[len(v["ms"]) // 2]
    return {"table_bytes_x2_4": total, "modes": res}


def search_modes(rounds):
    from skder_b200 import engine, synth

    packed = synth.config_packed("config4", engine.pack_contigs)
    db, queries = packed[:-64], packed[-64:]
    out = {"db_genomes": len(db), "queries": len(queries)}
    with engine.Engine(0) as eng:
        eng.add(db)
        eng.index()
        total = table_bytes(eng, 4)
        modes = {"resident": None, "on_demand": total / 8 / MIB}
        res = {m: {"ms": []} for m in modes}
        for r in range(rounds + 1):
            for m in (list(modes) if r % 2 else list(modes)[::-1]):
                with budget(modes[m]):
                    eng.index()
                    eng.search(queries, screen=80.0, min_af=15.0)  # steady state, as a resident daemon serves
                    (hits, st), ms, launches = timed(eng, lambda: eng.search(queries, screen=80.0, min_af=15.0))
                    on, blocks = eng.table_blocks()
                if r:
                    res[m]["ms"].append(round(ms, 1))
                res[m].update(on_demand=on, blocks=blocks, launches=launches, hits=len(hits), hits_sha256=sha(hits))
    assert len({v["hits_sha256"] for v in res.values()}) == 1, res
    for v in res.values():
        v["median_ms"] = sorted(v["ms"])[len(v["ms"]) // 2]
    out.update(table_bytes_x2_4=total, modes=res)
    return out


def capacity(src, copies):
    """src: the indexed config3 context; its sketches imported `copies` times into a second context"""
    import torch
    from skder_b200 import engine

    n = src.n_genomes
    rng = np.random.default_rng(7)
    qids = np.sort(rng.choice(n, 64, replace=False)).astype(np.int32)
    src.set_max_results(0)
    want, _ = src.rect(np.arange(n, dtype=np.int32), qids, screen=80.0, min_af=15.0)
    v = src.sketch_view()
    seeds_total = int(v.n_seeds)
    out = {"copies": copies, "genomes": n * copies, "seeds": seeds_total * copies,
           "resident_bytes_x2_1_per_layout": None}
    free0, total_b = torch.cuda.mem_get_info(0)
    with engine.Engine(0) as big:
        t0 = time.perf_counter()
        for _ in range(copies):
            rc = big._L.skb_import_sketches(big._h, v.n_genomes, v.dev_seeds, v.n_seeds, v.dev_marker_keys,
                                            v.n_marker_keys, v.host_seed_off, v.host_total_len, v.host_ctg_off,
                                            v.host_ctg_len, 0)
            big._ck(rc, "skb_import_sketches")
        n_db = big.n_genomes
        big.index()
        t_index = time.perf_counter() - t0
        on, _ = big.table_blocks()
        free1, _ = torch.cuda.mem_get_info(0)
        # seed records 8 B, marker structures (raw keys, inverted index, per-genome lists) 24 B per marker, tables at
        # the densest resident density 16 B per seed (DESIGN.md section 2)
        n_mk = int(v.n_marker_keys) * copies
        resident = seeds_total * copies * (8 + 16) + n_mk * 24
        out.update(index_s=round(t_index, 1), on_demand=on, device_bytes=total_b, free_before=free0,
                   free_after_index=free1, resident_bytes_x2_1_per_layout=resident,
                   resident_exceeds_device=resident > total_b)
        refs = np.arange(n_db, dtype=np.int32)
        big.timer_start()
        try:
            got, st = big.rect(refs, qids, screen=80.0, min_af=15.0)
        except Exception as e:
            out.update(error=str(e), free_at_error=torch.cuda.mem_get_info(0)[0])
            print(json.dumps(out), flush=True)
            raise
        out["search_ms"] = round(big.timer_stop(), 1)
        out["blocks"] = big.table_blocks()[1]
        out["hits"] = len(got)
        out["pairs_screened"] = int(st.n_pairs_screened)
        # a query q of the original set is genome q of every copy too; its hit on copy c of r is r + c * n.  Its own
        # copies are hits of their own (ANI 100), which the original set has no genome for.
        ok = True
        for q in qids.tolist():
            w = want[want["b"] == q]
            g = got[got["b"] == q]
            g = g[(g["a"] % n) != q]
            exp = np.sort(np.concatenate([w["a"].astype(np.int64) + c * n for c in range(copies)]))
            if not (np.array_equal(np.sort(g["a"].astype(np.int64)), exp)):
                ok = False
                break
            for c in range(copies):
                gc = g[(g["a"] // n) == c]
                if not (np.array_equal(gc["ani"], w["ani"]) and np.array_equal(gc["af_a"], w["af_a"])
                        and np.array_equal(gc["af_b"], w["af_b"])):
                    ok = False
                    break
        out["hits_equal_original_per_copy"] = ok
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--copies", type=int, default=36)
    ap.add_argument("--skip-triangle", action="store_true")
    ap.add_argument("--skip-capacity", action="store_true")
    ap.add_argument("--skip-search", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    from skder_b200 import engine, synth

    res = {"card": card(0)}
    t0 = time.perf_counter()
    packed = synth.config_packed("config3", engine.pack_contigs)
    eng = engine.Engine(0)
    eng.add(packed)
    del packed
    eng.index()
    res["config3_setup_s"] = round(time.perf_counter() - t0, 1)
    if not a.skip_triangle:
        res["triangle"] = triangle_modes(eng, a.rounds)
    if not a.skip_search:
        res["search"] = search_modes(a.rounds)
    if not a.skip_capacity:
        res["capacity"] = capacity(eng, a.copies)
    eng.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
