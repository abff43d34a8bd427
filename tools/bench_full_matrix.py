"""skani's `triangle --full-matrix` output (DESIGN.md section 3) on the config3 workload on one GPU.

  python tools/bench_full_matrix.py [--workload config3] [--rounds 2] [--dir /dev/shm] [--out result.json]

config3 is bench.py's default workload: 5,000 synthetic genomes of 5 Mbp (100 clades of 50), triangle at bench.py's
-s 89.5 --min-af 50.  Reported, with the card's name, power limit and max SM clock read in the same run:
- the triangle: skb_stats' device time and the wall time of Engine.triangle;
- per matrix (ANI, distance, AF), in a profiled pass of its own (torch.profiler, CUDA activities): the device time of the
  render (the matrix kernels, the row scan and the map memsets) and of the device-to-host copies, and the copy rate;
- per matrix, unprofiled and alternated over --rounds: the wall time of Engine.write_matrix to a finished file in --dir,
  and of Python rendering the same host edges into the same file (`%.2f` per cell, joined rows), the two files
  asserted byte-identical.
Prints one JSON line.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_estimators import build_engine, card  # noqa: E402

KINDS = ("ani", "distance", "af")


def python_render(n, labels, edges, kind):
    """the matrix file as bytes, formatted by Python from the host edge list"""
    a, b = edges["a"].astype(np.int64), edges["b"].astype(np.int64)
    m = np.full((n, n), "100.00" if kind == "distance" else "0.00", object)
    if kind == "af":
        m[a, b] = ["%.2f" % x for x in edges["af_a"].tolist()]
        m[b, a] = ["%.2f" % x for x in edges["af_b"].tolist()]
    else:
        t = ["%.2f" % x for x in edges["ani"].tolist()]
        if kind == "distance":
            t = ["%d.%02d" % divmod(10000 - int(x.replace(".", "")), 100) for x in t]
        m[a, b] = m[b, a] = t
    np.fill_diagonal(m, "0.00" if kind == "distance" else "100.00")
    return ("%d\n" % n + "".join(lb + "\t" + "\t".join(row) + "\n" for lb, row in zip(labels, m.tolist()))).encode()


def profiled_render(eng, path, labels, kind):
    """(render device ms, device-to-host copy ms) of one write_matrix, from torch.profiler's CUDA activities"""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.write_matrix(path, labels, kind)
    render = copy = 0.0
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if "Memcpy DtoH" in ev.key:
            copy += us / 1000
        elif "Memcpy" not in ev.key:
            render += us / 1000
    return render, copy


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config3")
    ap.add_argument("--screen", type=float, default=89.5)
    ap.add_argument("--min-af", type=float, default=50.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    ap.add_argument("--out")
    a = ap.parse_args()
    import torch

    res = {"card": card(0), "workload": a.workload, "screen": a.screen, "min_af": a.min_af}
    eng, n, t_setup = build_engine(a.workload, 0)
    res.update(genomes=n, setup_s=round(t_setup, 1))
    labels = ["genomes/clade%03d_member%03d.fasta" % (i // 50, i % 50) for i in range(n)]
    eng.triangle(screen=a.screen, min_af=a.min_af)  # warm-up
    t0 = time.perf_counter()
    edges, st = eng.triangle(screen=a.screen, min_af=a.min_af)
    res["triangle"] = {"wall_ms": round((time.perf_counter() - t0) * 1e3, 1), "device_ms": round(st.ms_total, 1),
                       "edges": int(st.n_edges)}
    torch.cuda.init()
    with tempfile.TemporaryDirectory(prefix="bench_full_matrix.", dir=a.dir) as tmp:
        gpu_path, py_path = os.path.join(tmp, "gpu.txt"), os.path.join(tmp, "py.txt")
        for kind in KINDS:  # warm-up: the kernels, CUB's scan, the pinned buffers
            eng.write_matrix(gpu_path, labels, kind)
        prof = {}
        for kind in KINDS:
            render_ms, copy_ms = profiled_render(eng, gpu_path, labels, kind)
            size = os.path.getsize(gpu_path)
            prof[kind] = {"bytes": size, "render_device_ms": round(render_ms, 2), "copy_dtoh_ms": round(copy_ms, 2),
                          "copy_gb_s": round(size / copy_ms / 1e6, 1) if copy_ms else None}
        res["profiled"] = prof
        walls = {k: {"gpu_s": [], "python_s": []} for k in KINDS}
        for _ in range(a.rounds):
            for kind in KINDS:
                t0 = time.perf_counter()
                eng.write_matrix(gpu_path, labels, kind)
                walls[kind]["gpu_s"].append(round(time.perf_counter() - t0, 3))
                t0 = time.perf_counter()
                text = python_render(n, labels, edges, kind)
                with open(py_path, "wb") as f:
                    f.write(text)
                walls[kind]["python_s"].append(round(time.perf_counter() - t0, 3))
                with open(gpu_path, "rb") as f:
                    assert f.read() == text, kind
                del text
        res["wall"] = walls
        res["identical"] = True
        res["dir"] = a.dir or tempfile.gettempdir()
    eng.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
