"""`skani triangle` from the FASTAs against the same triangle from `sketch -o DB`'s DB/*.sketch files (DESIGN.md
sections 3 and 5) on the config3 workload on one GPU.

  python tools/bench_sketch_inputs.py [--workload config3] [--rounds 2] [--dir /dev/shm] [--out result.json]

config3 is bench.py's default workload: 5,000 synthetic genomes of 5 Mbp (100 clades of 50), written as FASTA under
--dir, compared at bench.py's greedy thresholds (-s 89.5 --min-af 50).  Reported, with the card's name and power limit
read in the same run:
- the shim's `sketch -l LIST -o DB` wall time, and what writing the 5,000 descriptors costs of it;
- the shim's `triangle -E` wall time and its phases (SKB_PHASE_LOG) from the FASTA list and from a list of the
  DB/*.sketch files, alternated over --rounds; the two TSVs are asserted byte-identical (their SHA-256 is reported);
- the device time of skb_db_load_genomes' key-selection kernels (torch.profiler, CUDA activities) for all genomes
  requested in the triangle's order, and that call's wall time;
- the descriptor writing on config4's 20,000 genomes: sketch_files.write_all reads only the database's header, host
  tables and manifest, so it is timed on a database with config4's genome count and contig tables (one contig per
  genome: config4 genomes are single-contig) and its manifest, without the seed payload it never reads.
Prints one JSON line.
"""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from multiprocessing import Pool

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_estimators import card  # noqa: E402

SHIM = os.path.join(ROOT, "skder_b200", "bin", "skani")
SCREEN, MIN_AF = "89.5", "50"
KEY_KERNELS = ("db_key_runs_kernel", "db_key_counts_kernel", "db_select_keys_kernel")


def write_fastas(workload, d, procs):
    from bench import _write_clade_fasta
    from skder_b200 import synth

    nc, per = synth.CONFIGS[workload][:2]
    with Pool(procs) as p:
        p.map(_write_clade_fasta, [(workload, c, per, d) for c in range(nc)])
    return [os.path.join(d, "clade%03d_member%03d.fasta" % (c, m)) for c in range(nc) for m in range(per)]


def shim(argv, env=None):
    t0 = time.perf_counter()
    r = subprocess.run([sys.executable, SHIM] + argv, capture_output=True, env=dict(os.environ, SKB_NO_DAEMON="1", **(env or {})))
    wall = time.perf_counter() - t0
    if r.returncode:
        raise RuntimeError("%s: %s" % (argv[:2], r.stderr.decode()[-2000:]))
    return wall


def triangle(lst, out, threads):
    wall = shim(["triangle", "-l", lst, "-E", "-s", SCREEN, "--min-af", MIN_AF, "-t", str(threads), "-o", out],
                {"SKB_PHASE_LOG": "1"})
    with open(out, "rb") as f:
        sha = hashlib.sha256(f.read()).hexdigest()
    with open(out + ".skani_b200.phases.json") as f:
        ph = json.load(f)
    return {"wall_s": round(wall, 3), "phases": {k: round(v, 3) if isinstance(v, float) else v for k, v in ph.items()},
            "tsv_sha256": sha}


def key_kernels(db, ids):
    """(device ms of the key-selection kernels and of the whole call by kind, wall ms) of one load_genomes"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    from skder_b200 import engine

    torch.cuda.init()
    with engine.Engine(0) as eng:
        eng.load_genomes(db, ids)  # warm-up: module load, CUB's scan, scratch sizes
        eng.pop_last_add()
        t0 = time.perf_counter()
        eng.load_genomes(db, ids)
        wall = (time.perf_counter() - t0) * 1e3
        eng.pop_last_add()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.load_genomes(db, ids)
    dev = {"kernels": {}, "scan_ms": 0.0, "h2d_ms": 0.0}
    for ev in prof.key_averages():
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if ev.key in KEY_KERNELS:
            dev["kernels"][ev.key] = round(us / 1e3, 3)
        elif "Scan" in ev.key:
            dev["scan_ms"] += us / 1e3
        elif "Memcpy HtoD" in ev.key:
            dev["h2d_ms"] += us / 1e3
    dev["scan_ms"], dev["h2d_ms"] = round(dev["scan_ms"], 3), round(dev["h2d_ms"], 1)
    dev["selection_ms"] = round(sum(dev["kernels"].values()) + dev["scan_ms"], 3)
    return dev, round(wall, 1)


def descriptor_cost_config4(tmp):
    """seconds of sketch_files.write_all for config4's 20,000 genomes (see the module docstring)"""
    import struct

    from skder_b200 import cli, sketch_files, synth

    nc, per, length = synth.CONFIGS["config4"][:3]
    n = nc * per
    d = os.path.join(tmp, "config4_db")
    os.makedirs(d)
    with open(os.path.join(d, "sketches.skb"), "wb") as f:
        f.write(b"SKB200v1" + struct.pack("<4Q", n, 0, 0, n) + np.zeros(n + 1, "<u8").tobytes()
                + np.full(n, length, "<u8").tobytes() + np.arange(n + 1, dtype="<u4").tobytes()
                + np.full(n, length, "<u4").tobytes())
    paths = [os.path.join(tmp, "genomes", "clade%03d_member%03d.fasta" % (c, m)) for c in range(nc) for m in range(per)]
    names = ["c%d_m%d_ctg0" % (c, m) for c in range(nc) for m in range(per)]
    cli.write_atomic(os.path.join(d, "manifest.json"), json.dumps({"paths": paths, "names": names}))
    t0 = time.perf_counter()
    sketch_files.write_all(d, paths, paths, names, False, cli.write_atomic)
    return n, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config3")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--threads", type=int, default=min(32, os.cpu_count() or 1))
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out")
    a = ap.parse_args()
    res = {"card": card(0), "workload": a.workload, "screen": float(SCREEN), "min_af": float(MIN_AF),
           "threads": a.threads, "dir": a.dir or tempfile.gettempdir()}
    tmp = tempfile.mkdtemp(prefix="bench_sketch_inputs.", dir=a.dir)
    try:
        from skder_b200 import cli, sketch_files

        t0 = time.perf_counter()
        os.makedirs(os.path.join(tmp, "genomes"))
        fastas = write_fastas(a.workload, os.path.join(tmp, "genomes"), a.threads)
        res["genomes"] = len(fastas)
        res["write_fasta_s"] = round(time.perf_counter() - t0, 1)
        res["fasta_gb"] = round(sum(os.path.getsize(p) for p in fastas) / 1e9, 2)
        fl = os.path.join(tmp, "fastas.txt")
        with open(fl, "w") as f:
            f.write("".join(p + "\n" for p in fastas))
        db = os.path.join(tmp, "db")
        res["sketch_wall_s"] = round(shim(["sketch", "-l", fl, "-o", db, "-t", str(a.threads)]), 3)
        with open(os.path.join(db, "manifest.json")) as f:
            man = json.load(f)
        t0 = time.perf_counter()  # the descriptors again, timed on their own (same bytes)
        sketch_files.write_all(db, fastas, man["paths"], man["names"], False, cli.write_atomic)
        res["sketch_descriptors_s"] = round(time.perf_counter() - t0, 3)
        res["db_bytes"] = {"sketches.skb": os.path.getsize(os.path.join(db, "sketches.skb")),
                           "manifest.json": os.path.getsize(os.path.join(db, "manifest.json"))}
        names = sketch_files.file_names(fastas)
        sl = os.path.join(tmp, "sketches.txt")
        with open(sl, "w") as f:
            f.write("".join(os.path.join(db, names[p]) + "\n" for p in fastas))
        runs = {"fasta": [], "sketch": []}
        for _ in range(a.rounds):
            for kind, lst in (("fasta", fl), ("sketch", sl)):
                runs[kind].append(triangle(lst, os.path.join(tmp, kind + ".tsv"), a.threads))
        shas = {r["tsv_sha256"] for k in runs for r in runs[k]}
        assert len(shas) == 1, shas
        res["tsv_sha256"] = shas.pop()
        res["edges"] = runs["fasta"][0]["phases"]["edges"]
        res["triangle"] = runs
        order = {p: i for i, p in enumerate(man["paths"])}
        res["load_genomes"], res["load_genomes_wall_ms"] = key_kernels(db, [order[p] for p in sorted(fastas)])
        n4, s4 = descriptor_cost_config4(tmp)
        res["config4_descriptors"] = {"genomes": n4, "write_all_s": round(s4, 3)}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
