"""Cost of skani's -m marker compression (DESIGN.md section 3) on a synthetic workload (default config3: 5,000 genomes x
5 Mbp) on one GPU, at m = 1000 (the default), 500 and 200.

  python tools/bench_marker_c.py [--workload config3] [--ms 1000,500,200] [--rounds 5] [--out result.json]

The genomes are generated and packed once.  For every m a context of its own sketches them (upload + sketch, host clock
around skb_add_genomes, which returns after the last batch is sketched) and indexes them (CUDA events on the library's
stream; seed and chunk tables do not depend on m, so the differences between the m values are the marker sort's).
Every round then times one resident triangle per m (bench.py's skDER greedy settings: -s 89.5, --min-af 50) with CUDA
events, the m that goes first rotating; the library's own screen time (skb_stats.ms_screen) is reported beside it.
Per m: raw marker keys, pairs that pass the screen, edges and bench.py's edges_sha256 of them.  The card's name and
power limit are read in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_estimators import card  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config3")
    ap.add_argument("--ms", default="1000,500,200")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out")
    args = ap.parse_args()
    import numpy as np

    import bench
    from skder_b200 import engine, synth

    ms = [int(x) for x in args.ms.split(",")]
    t0 = time.perf_counter()
    packed = synth.config_packed(args.workload, engine.pack_contigs)
    n = len(packed)
    t_gen = time.perf_counter() - t0
    engines, res = {}, {}
    for m in ms:
        eng = engine.Engine(args.device)
        eng.set_marker_compression(m)
        t1 = time.perf_counter()
        eng.add(packed)
        t_sketch = time.perf_counter() - t1
        eng.timer_start()
        eng.index()
        res[m] = {"sketch_s": round(t_sketch, 3), "index_ms": round(eng.timer_stop(), 2),
                  "marker_keys": int(eng.sketch_view().n_marker_keys), "triangle_ms": [], "screen_ms": []}
        engines[m] = eng
    for m in ms:  # warm-up: every context's kernels and scratch sizes
        engines[m].triangle(bench.GREEDY_SCREEN, bench.GREEDY_MIN_AF)
    for r in range(args.rounds):
        for m in ms[r % len(ms):] + ms[:r % len(ms)]:
            eng = engines[m]
            eng.timer_start()
            edges, st = eng.triangle(bench.GREEDY_SCREEN, bench.GREEDY_MIN_AF)
            res[m]["triangle_ms"].append(round(eng.timer_stop(), 2))
            res[m]["screen_ms"].append(round(st.ms_screen, 2))
            res[m].update(pairs_total=st.n_pairs_total, pairs_screened=st.n_pairs_screened, edges=len(edges),
                          edges_sha256=bench.canonical_edges(edges, np.arange(n)))
    for m in ms:
        engines[m].close()
        for k in ("triangle_ms", "screen_ms"):
            res[m][k + "_median"] = sorted(res[m][k])[len(res[m][k]) // 2]
        res[m]["pairs_per_s"] = round(res[m]["pairs_total"] / (res[m]["triangle_ms_median"] / 1e3))
    out = {"workload": args.workload, "genomes": n, "generate_s": round(t_gen, 1), "screen": bench.GREEDY_SCREEN,
           "min_af": bench.GREEDY_MIN_AF, "card": card(args.device), "m": {str(m): res[m] for m in ms}}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
