"""Resident triangle of a synthetic workload (default config3: 5,000 genomes x 5 Mbp) in the three ANI estimator modes
(skani's default mean, --median, --robust; DESIGN.md section 3), alternated round by round on one GPU.

  python tools/bench_estimators.py [--workload config3] [--rounds 5] [--out result.json]

The sketch DB is built and indexed once; every round then times one skb_triangle per mode with CUDA events on the
library's stream (Engine.timer_start / timer_stop), modes in rotating order.  A second process with SKB_TRACE=1 runs
one triangle per mode and reports the per-batch `estimator` span (and the `finalize` span beside it) from the library's
trace; tracing records extra events, so it is kept out of the timed process.  The card's name and power limit are read
in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
MODES = ("mean", "median", "robust")
SCREEN, MIN_AF = 80.0, 15.0  # skder's greedy defaults, as bench.py runs them


def build_engine(workload, device):
    from skder_b200 import engine, synth

    t0 = time.perf_counter()
    packed = synth.config_packed(workload, engine.pack_contigs)
    eng = engine.Engine(device)
    eng.add(packed)
    eng.index()
    return eng, len(packed), time.perf_counter() - t0


def card(device):
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm",
                                       "--format=csv,noheader"], text=True, timeout=30).strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clk}
    except (OSError, subprocess.SubprocessError, ValueError) as e:
        return {"error": str(e)}


def timed(args):
    eng, n, t_setup = build_engine(args.workload, args.device)
    res = {m: [] for m in MODES}
    stats = {}
    for m in MODES:  # warm-up: every mode's kernels, CUB's algorithm choice and the scratch sizes
        eng.set_estimator(m)
        eng.triangle(SCREEN, MIN_AF)
    for r in range(args.rounds):
        for m in MODES[r % 3:] + MODES[:r % 3]:
            eng.set_estimator(m)
            l0 = eng.launches
            eng.timer_start()
            edges, st = eng.triangle(SCREEN, MIN_AF)
            res[m].append(eng.timer_stop())
            stats[m] = {"pairs_total": st.n_pairs_total, "pairs_screened": st.n_pairs_screened, "edges": len(edges),
                        "launches": eng.launches - l0}
    eng.close()
    out = {"workload": args.workload, "genomes": n, "setup_s": round(t_setup, 1), "card": card(args.device), "modes": {}}
    for m in MODES:
        ms = sorted(res[m])
        med = ms[len(ms) // 2]
        out["modes"][m] = dict(stats[m], ms=[round(x, 2) for x in res[m]], ms_median=round(med, 2),
                               pairs_per_s=round(stats[m]["pairs_total"] / (med / 1e3)),
                               screened_pairs_per_s=round(stats[m]["pairs_screened"] / (med / 1e3)))
    return out


def traced(args):
    """child process (SKB_TRACE=1): one triangle per mode; the library writes the per-batch timeline on stderr"""
    eng, _, _ = build_engine(args.workload, args.device)
    for m in MODES:
        eng.set_estimator(m)
        sys.stderr.write("@@mode warm-up\n")
        eng.triangle(SCREEN, MIN_AF)
        sys.stderr.write("@@mode %s\n" % m)
        sys.stderr.flush()
        eng.triangle(SCREEN, MIN_AF)
        sys.stderr.flush()
    eng.close()


def spans(args):
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--traced", "--workload", args.workload, "--device",
                        str(args.device)], env=dict(os.environ, SKB_TRACE="1"), capture_output=True, text=True)
    if p.returncode:
        return {"error": p.stderr[-2000:]}
    out, mode = {m: {} for m in MODES}, None
    for line in p.stderr.splitlines():
        if line.startswith("@@mode"):
            mode = line.split()[1]
            continue
        t = re.match(r"\[skb trace\] batch (\d+) (\w+) .*\(([\d.]+)\)", line)
        if mode in out and t and t.group(2) in ("finalize", "estimator"):
            out[mode].setdefault(t.group(2) + "_ms_per_batch", []).append(float(t.group(3)))
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
