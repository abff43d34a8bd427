"""Resident triangle of a synthetic workload (default config3: 5,000 genomes x 5 Mbp) with skani's --detailed columns
off and on (DESIGN.md section 3), alternated round by round on one GPU.

  python tools/bench_detail.py [--workload config3] [--rounds 5] [--out result.json]

The sketch DB is built and indexed once; every round then times one skb_triangle per setting with CUDA events on the
library's stream (Engine.timer_start / timer_stop), the setting that goes first alternating.  The "on" time includes
copying the detail records to the host (Engine.last_edge_detail), as the shim does; the contig statistics are host-only
and not timed.  A second process with SKB_TRACE=1 runs one triangle per setting and reports the per-batch `detail` span
(sd_kernel) and the `ci` and `finalize` spans beside it from the library's trace; tracing records extra events, so it
is kept out of the timed process.  The card's name and power limit are read in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import re
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_estimators import SCREEN, MIN_AF, build_engine, card  # noqa: E402

SETTINGS = ("off", "on")


def run(eng, setting):
    eng.set_detailed(setting == "on")
    edges, st = eng.triangle(SCREEN, MIN_AF)
    det = eng.last_edge_detail() if setting == "on" else None
    return edges, st, det


def timed(args):
    eng, n, t_setup = build_engine(args.workload, args.device)
    res = {s: [] for s in SETTINGS}
    stats = {}
    for s in SETTINGS:  # warm-up: both paths' kernels and scratch sizes
        run(eng, s)
    for r in range(args.rounds):
        for s in SETTINGS[r % 2:] + SETTINGS[:r % 2]:
            l0 = eng.launches
            eng.timer_start()
            edges, st, det = run(eng, s)
            res[s].append(eng.timer_stop())
            stats[s] = {"pairs_total": st.n_pairs_total, "pairs_screened": st.n_pairs_screened, "edges": len(edges),
                        "launches": eng.launches - l0}
            if det is not None and len(det):
                sd = det["sd"]
                stats[s]["sd_pp"] = {"median": round(float(sorted(sd)[len(sd) // 2]), 3), "max": round(float(sd.max()), 3)}
    eng.set_detailed(False)
    eng.close()
    out = {"workload": args.workload, "genomes": n, "setup_s": round(t_setup, 1), "card": card(args.device), "detailed": {}}
    for s in SETTINGS:
        ms = sorted(res[s])
        med = ms[len(ms) // 2]
        out["detailed"][s] = dict(stats[s], ms=[round(x, 2) for x in res[s]], ms_median=round(med, 2),
                                  pairs_per_s=round(stats[s]["pairs_total"] / (med / 1e3)))
    return out


def traced(args):
    """child process (SKB_TRACE=1): one triangle per setting; the library writes the per-batch timeline on stderr"""
    eng, _, _ = build_engine(args.workload, args.device)
    for s in SETTINGS:
        sys.stderr.write("@@setting warm-up\n")
        run(eng, s)
        sys.stderr.write("@@setting %s\n" % s)
        sys.stderr.flush()
        run(eng, s)
        sys.stderr.flush()
    eng.close()


def spans(args):
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--traced", "--workload", args.workload, "--device",
                        str(args.device)], env=dict(os.environ, SKB_TRACE="1"), capture_output=True, text=True)
    if p.returncode:
        return {"error": p.stderr[-2000:]}
    out, setting = {s: {} for s in SETTINGS}, None
    for line in p.stderr.splitlines():
        if line.startswith("@@setting"):
            setting = line.split()[1]
            continue
        t = re.match(r"\[skb trace\] batch (\d+) (\w+) .*\(([\d.]+)\)", line)
        if setting in out and t and t.group(2) in ("finalize", "ci", "detail"):
            out[setting].setdefault(t.group(2) + "_ms_per_batch", []).append(float(t.group(3)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config3")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out")
    ap.add_argument("--traced", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.traced:
        traced(args)
        return
    res = timed(args)
    res["trace"] = spans(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
