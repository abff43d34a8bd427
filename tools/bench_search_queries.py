"""Several queries per `skani search`, and the cost of -n (DESIGN.md section 3), on synthetic workloads on one GPU.

  python tools/bench_search_queries.py [--qs 1,16,64] [--rounds 3] [--cut-workload config3] [--out result.json]

Search: a database of 200 genomes (20 clades x 10, 1 Mbp, 0.05-2.5 % apart) is sketched through the shim, and 80
held-out members of the same clades are the queries.  For every Q the shim's `search` answers Q queries in one launch
(one Engine.search in the database's daemon) and, alternated with it, in Q launches of one query each; host clock
around the launches, the daemon started and warmed before the first timed round.  Reported: seconds per round and
searches/s of both.

-n: config3's generator (5 Mbp genomes), 4 clades x 250 members, split into references (even ids) and queries (odd
ids) and compared at -s 50, so that every query has about 125 edges.  The same skb_rect runs with -n 0 and -n 1,
alternated; the stage's time is the CUDA-event time the library adds to skb_stats.ms_total beyond ms_screen + ms_ani.
The card's name and power limit are read in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_estimators import card  # noqa: E402

SHIM = os.path.join(ROOT, "skder_b200", "bin", "skani")


def shim(argv, env):
    subprocess.run([sys.executable, SHIM] + argv, env=env, check=True, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL)


def bench_search(qs, rounds, device, tmp):
    from skder_b200 import daemon, synth

    db_paths, q_paths = [], []
    for c, k, contigs in synth.clade_genomes(20, 14, 1_000_000, 20261023, d_lo=0.0005, d_hi=0.025, max_contigs=50):
        p = os.path.join(tmp, "c%02d_%02d.fasta" % (c, k))
        synth.write_fasta(p, contigs, name="c%02d_%02d" % (c, k))
        (db_paths if k < 10 else q_paths).append(p)
    lst, db = os.path.join(tmp, "db.txt"), os.path.join(tmp, "db")
    with open(lst, "w") as f:
        f.write("".join(p + "\n" for p in db_paths))
    env = dict(os.environ, SKB_DEVICE=str(device), SKB_DAEMON_IDLE="600")
    env.pop("SKB_NO_DAEMON", None)
    out = os.path.join(tmp, "out.tsv")
    shim(["sketch", "-l", lst, "-o", db, "-t", "8"], env)
    res = {}
    try:
        shim(["search"] + q_paths[:max(qs)] + ["-d", db, "-o", out], env)  # starts and warms the daemon
        for q in qs:
            one, each = [], []
            for _ in range(rounds):
                t0 = time.perf_counter()
                shim(["search"] + q_paths[:q] + ["-d", db, "-o", out], env)
                one.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                for p in q_paths[:q]:
                    shim(["search", p, "-d", db, "-o", out], env)
                each.append(time.perf_counter() - t0)
            m1, me = sorted(one)[len(one) // 2], sorted(each)[len(each) // 2]
            res[str(q)] = {"one_launch_s": [round(x, 3) for x in one], "q_launches_s": [round(x, 3) for x in each],
                           "one_launch_searches_per_s": round(q / m1, 1), "q_launches_searches_per_s": round(q / me, 1)}
    finally:
        daemon.stop_for(db)
    return {"db_genomes": len(db_paths), "genome_bp": 1_000_000, "rounds": rounds, "q": res}


def bench_cut(workload, rounds, device):
    import numpy as np

    from skder_b200 import engine, synth

    packed = synth.config_packed(workload, engine.pack_contigs, n_clades=4, per_clade=250)
    n = len(packed)
    refs, queries = np.arange(0, n, 2), np.arange(1, n, 2)
    res = {"0": [], "1": []}
    with engine.Engine(device) as eng:
        eng.add(packed)
        eng.index()
        for n_max in (0, 1):  # warm-up of both shapes
            eng.set_max_results(n_max)
            eng.rect(refs, queries, screen=50.0, min_af=15.0)
        for r in range(rounds):
            for n_max in ((0, 1) if r % 2 == 0 else (1, 0)):
                eng.set_max_results(n_max)
                edges, st = eng.rect(refs, queries, screen=50.0, min_af=15.0)
                res[str(n_max)].append({"edges": len(edges), "ms_screen": round(st.ms_screen, 3),
                                        "ms_ani": round(st.ms_ani, 3),
                                        "ms_best_n": round(st.ms_total - st.ms_screen - st.ms_ani, 3),
                                        "launches": st.launches})
    stage = sorted(x["ms_best_n"] for x in res["1"])
    return {"workload": workload, "genomes": n, "refs": len(refs), "queries": len(queries), "screen": 50.0,
            "edges_all": res["0"][0]["edges"], "edges_n1": res["1"][0]["edges"],
            "best_n_ms_median": stage[len(stage) // 2], "runs": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--qs", default="1,16,64")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cut-workload", default="config3")
    ap.add_argument("--cut-rounds", type=int, default=6)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out")
    args = ap.parse_args()
    out = {"card": card(args.device)}
    with tempfile.TemporaryDirectory(prefix="skb-bench-") as tmp:
        out["search"] = bench_search([int(x) for x in args.qs.split(",")], args.rounds, args.device, tmp)
    out["best_n"] = bench_cut(args.cut_workload, args.cut_rounds, args.device)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
