#!/usr/bin/env python3
"""bench.py -- genome pairs/sec for ANI+AF behind skDER's `skani` call sites, and dereplication wall time.

  python bench.py --gpus N --steps K --warmup W            (ours; one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --steps K --warmup W    (CPU arm: the oracle port on all host threads)
  python bench.py --workload config2|config3|config3r|config4|config5 ...
  python bench.py ... --dump-outputs DIR                   (also write what the last timed step computed, as .npy)

A step = one pass of the hot path over one synthetic genome set (BASELINE.json configs):
  value : pairs/s with sketches already resident in HBM (prescreen + ANI/AF + edge gather), device-timed
  e2e   : pairs/s through the C-ABI from packed genomes in pinned HOST memory to edges on the host
          (H2D upload + sketch + index + prescreen + ANI/AF + D2H), every step.
  derep : wall seconds of the UNMODIFIED reference `skder -d greedy|dynamic` (baseline/_ref) on the same genomes
          written as FASTA files, with skder_b200/bin/skani first on PATH (N=1, triangle workloads).
config4 (`low_mem_greedy`) is the search path: a step = the greedy loop of reference src/skDER/skder.py:116-133
(one `skani search` per not-yet-accounted genome in N50 order) against the resident sketch database.
The default workload is the configuration BASELINE.json quotes its metric on (N=5k x 5 Mbp = configs[2], `config3`;
it fits one GPU).  N>1 shards the same triangle's rows over the ranks (no data-path collective; sketches are
replicated by NCCL all-gather before the timed region of `value`, inside it for `e2e`); seed tables are sharded by
reference genome (each rank builds and probes only its own genomes' tables) and the surviving pairs are exchanged once
(8 bytes per pair) between the prescreen and the ANI/AF stage.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GREEDY_SCREEN = 89.5  # skDER default: -s (ANI cutoff 99.5 - 10)   reference bin/skder:199-204 (greedy AND dynamic mode;
                      # dynamic lowers --min-af by 20 only together with -n, bin/skder:218-219)
GREEDY_MIN_AF = 50.0  # skDER default AF cutoff                    reference bin/skder:325-329
SEARCH_SCREEN, SEARCH_MIN_AF = 80.0, 15.0  # `skani search` defaults: skDER passes neither option (skder.py:119)
SKDER_ANI, SKDER_AF = 99.5, 50.0           # skDER's default cutoffs (bin/skder:96-97)
# bounded sample the `cpu_baseline` leg of OUR arm is timed on (same generator): 80 clades x 5 members keeps the
# workload's survivor fraction (1.0 % vs 0.98 %)
CPU_SAMPLE_CLADES, CPU_SAMPLE_PER_CLADE = 80, 5
SEARCH_BATCH_MAX = int(os.environ.get("SKB_SEARCH_BATCH", "64"))  # queries searched per call at most (1 = strictly one by one)
SEARCH_WORKLOADS = ("config4", "tiny4")  # low_mem_greedy: the `skani sketch` + `skani search` path
DUMP_MAX_BYTES = 64 << 20  # --dump-outputs writes at most this much


def cfg(name):
    from skder_b200 import synth

    return synth.CONFIGS[name]


def workload_shape(name):
    nc, per, L, Lhi, *_ = cfg(name)
    return nc, per, L


def workload_name(w):
    nc, per, L, Lhi, *_ = cfg(w)
    size = "%.1f Mbp" % (L / 1e6) if Lhi is None else "%.0f-%.0f Mbp" % (L / 1e6, Lhi / 1e6)
    if w in SEARCH_WORKLOADS:
        return ("%s: %d synthetic %s genomes (%d clades x %d), low_mem_greedy: `skani sketch` once, then the greedy loop of "
                "`skani search` calls (skani defaults -s 80 --min-af 15), skDER cutoffs 99.5 / 50" % (w, nc * per, size, nc, per))
    return ("%s: %d synthetic %s genomes (%d clades x %d, 95-99.9%% ANI within clade), skDER default thresholds: greedy and "
            "dynamic mode both run `skani triangle -s 89.5 --min-af 50 -E`" % (w, nc * per, size, nc, per))


class ClockSampler:
    """SM clock / throttle reasons sampled during the timed region: NVML from a thread of this process (pynvml), or an
    `nvidia-smi -lms` child where NVML is not importable.  NVML in-process keeps the polling light: every query takes
    a driver-wide lock, and an nvidia-smi loop per rank was seen to stall cudaMemGetInfo / cudaMalloc of the timed
    steps by tens of milliseconds."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    PERIOD = 0.25

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.th, self.stop = index, [], None, None, threading.Event()
        self.sm, self.mx, self.reasons = [], [], set()

    def __enter__(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            bits = {"hw_slowdown": pynvml.nvmlClocksThrottleReasonHwSlowdown,
                    "hw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": pynvml.nvmlClocksThrottleReasonSwThermalSlowdown,
                    "sw_power_cap": pynvml.nvmlClocksThrottleReasonSwPowerCap}
            self.mx.append(float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)))

            def poll():
                while True:
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.reasons.update(n for n, b in bits.items() if r & b)
                    except pynvml.NVMLError:
                        pass
                    if self.stop.wait(self.PERIOD):
                        return

            self.th = threading.Thread(target=poll, daemon=True)
            self.th.start()
            return self
        except Exception:
            self.th = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "250"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None
        return self

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [x for x in vis.split(",") if x.strip()]
        if ids and self.index < len(ids) and ids[self.index].strip().isdigit():
            return int(ids[self.index])
        return self.index

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.th.join(timeout=2)
        elif self.th:
            self.stop.set()
            self.th.join(timeout=2)

    def summary(self):
        if self.proc is None and self.sm:
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": [n for n in names if n in self.reasons], "samples": len(self.sm), "source": "nvml"}
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) >= 7 and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/skani_oracle.c) -- the reference's skani is not installable here
# ------------------------------------------------------------------------------------------------
def cpu_sketch_clades(workload, clades, per_clade, threads):
    """Oracle sketches of `clades` (ids) x per_clade members; returns (sketches, seconds spent sketching).  Genomes are
    generated clade by clade (not timed) so the ASCII text of a 5,000-genome workload is never resident at once."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle as O
    from skder_b200 import synth

    sk, t_sketch = [], 0.0
    with ThreadPoolExecutor(threads) as ex:
        step = max(1, threads // 4)
        for c0 in range(0, len(clades), step):
            gens = [g for cl in ex.map(lambda c: synth.clade_of(workload, c, per_clade), clades[c0:c0 + step]) for g in cl]
            t0 = time.perf_counter()
            sk += list(ex.map(O.Sketch.from_contigs, gens))
            t_sketch += time.perf_counter() - t0
    return sk, t_sketch


def cpu_triangle_components(workload, n_clades, per_clade, threads, screen, min_af):
    """One CPU pass over n_clades x per_clade genomes of the workload: sketching one genome per host thread, then the
    all-vs-all (inverted-index prescreen of every pair, ANI/AF of the survivors) inside the C library on `threads`
    pthreads (oracle/skani_oracle.c ora_triangle) -- no Python per pair."""
    from oracle import oracle as O

    O.build()
    sk, t_sketch = cpu_sketch_clades(workload, list(range(n_clades)), per_clade, threads)
    n = len(sk)
    r = O.triangle(sk, screen / 100.0, min_af / 100.0, threads)
    return {"n": n, "pairs": n * (n - 1) // 2, "survivors": r["survivors"], "edges": r["edges"], "t_sketch": t_sketch,
            "t_index": r["t_index"], "t_count": r["t_count"], "t_screen": r["t_index"] + r["t_count"], "t_ani": r["t_ani"]}


def cpu_extrapolate(comp, n_full, pairs_full, surv_full, with_sketch):
    # inverted-index prescreen: the key sort scales with the genomes, run counting with the shared markers (i.e. with
    # the surviving, within-clade pairs); ANI/AF with the surviving pairs
    t = (comp["t_count"] + comp["t_ani"]) / max(comp["survivors"], 1) * surv_full
    if with_sketch:  # end to end: sketching and the marker index are part of the step, as they are in our e2e
        t += (comp["t_sketch"] + comp["t_index"]) / comp["n"] * n_full
    return pairs_full / t, t


def cpu_search_loop(workload, threads, n_clades, per_clade):
    """config4 on the CPU: sketch every genome, then the greedy loop of skder.py:116-133 with one oracle `search`
    (screen + ANI/AF of the query against every database genome, on `threads` pthreads) per representative."""
    from oracle import oracle as O

    O.build()
    sk, t_sketch = cpu_sketch_clades(workload, list(range(n_clades)), per_clade, threads)
    n = len(sk)
    order = sorted(range(n), key=lambda g: (-n50_of(sk[g].contig_lens()), g))
    accounted, reps, rep_ids, t0 = set(), 0, [], time.perf_counter()
    for g in order:
        if g in accounted:
            continue
        reps += 1
        rep_ids.append(g)
        for r, ani, af_r, af_q in O.search(sk, g, SEARCH_SCREEN / 100.0, SEARCH_MIN_AF / 100.0, threads):
            if round(ani * 100, 2) >= SKDER_ANI and round(af_q * 100, 2) >= SKDER_AF:  # skder.py:128 (col 4 = the query's AF)
                accounted.add(r)
    return {"n": n, "reps": reps, "t_sketch": t_sketch, "t_loop": time.perf_counter() - t0, "reps_sha256": ids_sha256(rep_ids)}


def ids_sha256(ids):
    """checksum of a set of workload-wide genome numbers (the representatives of a search loop)"""
    import hashlib

    return hashlib.sha256(np.sort(np.asarray(list(ids), np.int64)).tobytes()).hexdigest()


def n50_of(lens):
    lens = np.sort(np.asarray(lens))[::-1]
    if len(lens) == 0:
        return 0
    c = np.cumsum(lens)
    return int(lens[np.searchsorted(c, int(c[-1] // 2))])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    nc, per, L = workload_shape(args.workload)
    n_full = nc * per
    if args.workload in SEARCH_WORKLOADS:
        return run_reference_search(args, threads)
    pairs_full = n_full * (n_full - 1) // 2
    surv_full = nc * per * (per - 1) // 2
    # warm-up on the bounded sample (threads, page cache, allocator); it is also the cross-check figure
    sample = None
    for _ in range(max(1, args.warmup)):
        sample = cpu_triangle_components(args.workload, min(nc, CPU_SAMPLE_CLADES), CPU_SAMPLE_PER_CLADE, threads, GREEDY_SCREEN,
                                         GREEDY_MIN_AF)
    x_value, x_t = cpu_extrapolate(sample, n_full, pairs_full, surv_full, with_sketch=True)
    # timed: --steps FULL passes over the workload itself
    comps = [cpu_triangle_components(args.workload, nc, per, threads, GREEDY_SCREEN, GREEDY_MIN_AF) for _ in range(args.steps)]
    t_steps = [c["t_sketch"] + c["t_screen"] + c["t_ani"] for c in comps]
    t_full = float(np.mean(t_steps))
    value = pairs_full / t_full
    c0 = comps[-1]
    sample_txt = ("the full workload, %d steps: %d genomes, %d pairs, %d survive the screen, "
                  "%d edges; per step: sketch %.2f s, inverted-index prescreen %.2f s, ANI/AF %.2f s on %d threads (genome generation "
                  "not timed)" % (len(comps), c0["n"], c0["pairs"], c0["survivors"], c0["edges"],
                                  float(np.mean([c["t_sketch"] for c in comps])), float(np.mean([c["t_screen"] for c in comps])),
                                  float(np.mean([c["t_ani"] for c in comps])), threads))
    line = {
        "impl": "reference", "metric": "genome pairs/sec ANI+AF", "value": value, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": len(comps), "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": t_full * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/int32 + f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload), "screen": GREEDY_SCREEN, "min_af": GREEDY_MIN_AF, "pairs": pairs_full,
                   "pairs_screened": c0["survivors"], "edges": c0["edges"],
                   "note": "oracle-CPU (C port of the published skani method), NOT the skani binary: skani is absent. "
                           "Warm-up steps run on a bounded sample; every timed step is the whole workload",
                   "sample_cross_check": {"genomes": sample["n"], "pairs": sample["pairs"], "survivors": sample["survivors"],
                                          "extrapolated_value": x_value, "extrapolated_ms_per_step": x_t * 1e3}},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": sample_txt},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def run_reference_search(args, threads):
    nc, per, L = workload_shape(args.workload)
    s_clades = min(nc, int(os.environ.get("SKB_REF_SEARCH_CLADES", "20")))
    for _ in range(args.warmup):
        cpu_search_loop(args.workload, threads, s_clades, per)
    runs = [cpu_search_loop(args.workload, threads, s_clades, per) for _ in range(args.steps)]
    r = runs[-1]
    t_sketch, t_loop = float(np.mean([x["t_sketch"] for x in runs])), float(np.mean([x["t_loop"] for x in runs]))
    # searches scale with representatives x database size: R ~ clades, each search touches N genomes' markers and
    # ~per same-clade survivors
    n_full = nc * per
    t_search = t_loop / r["reps"]
    t_full = t_sketch / r["n"] * n_full + (r["reps"] / s_clades * nc) * t_search * (n_full / r["n"])
    pairs = (r["reps"] / s_clades * nc) * n_full
    line = {
        "impl": "reference", "metric": "genome pairs/sec ANI+AF (search path)", "value": pairs / t_full, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": len(runs), "steps_requested": args.steps, "warmup": args.warmup, "ms_per_step": t_full * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/int32 + f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload),
                   "note": "oracle-CPU, NOT skani; EXTRAPOLATED from %d clades x %d (%d genomes, %d searches, %.2f s sketch + "
                           "%.2f s loop per step): sketching scales with genomes, the loop with representatives x database size"
                           % (s_clades, per, r["n"], r["reps"], t_sketch, t_loop)},
        "cpu_baseline": {"value": pairs / t_full, "unit": "pairs/s", "cores": threads, "kind": "port",
                         "sample": "%d clades x %d of %s, extrapolated" % (s_clades, per, args.workload)},
        "e2e": {"value": pairs / t_full, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# ours
# ------------------------------------------------------------------------------------------------
def pinned_views(packed, torch):
    """Copy every genome's 2-bit words into ONE pinned host buffer and return skb_packed views into it."""
    from skder_b200 import _lib

    total = sum(p.n_words for p in packed)
    pin = torch.empty(total, dtype=torch.int64).pin_memory()
    arr = pin.numpy().view(np.uint64)
    views, keep, off = [], [], 0
    for p in packed:
        nw = p.n_words
        arr[off:off + nw] = p.words()
        v = _lib.Packed()
        v.words = C.cast(arr[off:].ctypes.data, C.POINTER(C.c_uint64))
        v.n_words, v.n_bases, v.n_contigs = nw, p.n_bases, p.n_contigs
        lens = (C.c_int64 * max(1, p.n_contigs))(*p.contig_lens().tolist())
        v.contig_lens = C.cast(lens, C.POINTER(C.c_int64))
        v.first_name, v.n50, v.total_bases_all = None, p.n50, p.total_bases_all
        keep.append(lens)
        views.append(v)
        off += nw
    return pin, views, keep, total * 8


def canonical_table(edges, canon):
    """Edge records -> columns keyed by workload-wide genome numbers (clade * per + member), the lower number in `a`
    (AFs swapped with it), rows sorted by (a, b): the same whatever order the ranks ingested the genomes in."""
    a, b = canon[edges["a"]], canon[edges["b"]]
    sw = a > b
    lo, hi = np.where(sw, b, a), np.where(sw, a, b)
    af_lo, af_hi = np.where(sw, edges["af_b"], edges["af_a"]), np.where(sw, edges["af_a"], edges["af_b"])
    order = np.lexsort((hi, lo))
    return {"a": lo[order], "b": hi[order], "ani": edges["ani"][order], "af_a": af_lo[order], "af_b": af_hi[order]}


def canonical_edges(edges, canon):
    """sha256 of the canonical table as 2-decimal text rows: the same for every N if the results are."""
    t = canonical_table(edges, canon)
    h = hashlib.sha256()
    for row in zip(t["a"], t["b"], t["ani"], t["af_a"], t["af_b"]):
        h.update(b"%d\t%d\t%.2f\t%.2f\t%.2f\n" % row)
    return h.hexdigest()


def dump_outputs(directory, prefix, columns, max_bytes=DUMP_MAX_BYTES):
    """Columns of one output table -> DIR/<prefix>_<column>.npy in float64 (genome numbers are exact there); returns the
    bytes written.  A table above max_bytes keeps a fixed, seeded sample of its rows, the same rows for the same length."""
    os.makedirs(directory, exist_ok=True)
    n = len(next(iter(columns.values())))
    rows = np.arange(n)
    if n * 8 * len(columns) > max_bytes:
        rows = np.sort(np.random.default_rng(0).choice(n, max_bytes // (8 * len(columns)), replace=False))
    for name, col in columns.items():
        np.save(os.path.join(directory, "%s_%s.npy" % (prefix, name)), np.asarray(col, np.float64)[rows])
    return len(rows) * 8 * len(columns)


def parity_sample(workload, edges, per, n_clades_checked, n_each, threads, screen, min_af):
    """Outside every timed region: oracle verdicts for >= n_each pairs the GPU kept and >= n_each pairs it rejected, drawn
    from n_clades_checked whole clades of the bench's own workload (N=1: genome id = clade * per + member)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import oracle as O

    rng = np.random.default_rng(12345)
    nc = workload_shape(workload)[0]
    clades = sorted(rng.choice(nc, size=min(nc, n_clades_checked), replace=False).tolist())
    sk, _ = cpu_sketch_clades(workload, clades, per, threads)
    gid = {c * per + m: sk[k * per + m] for k, c in enumerate(clades) for m in range(per)}
    ids = np.array(sorted(gid))
    have = {(int(e["a"]), int(e["b"])): e for e in edges if int(e["a"]) in gid and int(e["b"]) in gid}
    kept = sorted(have)
    kept = [kept[i] for i in rng.choice(len(kept), size=min(n_each, len(kept)), replace=False)] if kept else []
    rejected = set()
    while len(rejected) < n_each and len(ids) > 1:
        a, b = sorted(rng.choice(ids, size=2, replace=False).tolist())
        if (a, b) not in have:
            rejected.add((a, b))
    rejected = sorted(rejected)

    def check_kept(ab):
        a, b = ab
        r = O.pair(gid[a], gid[b])
        ok = O.screen(gid[a], gid[b], screen / 100.0)[1] and r.ani >= 0 and max(r.af_a, r.af_b) * 100 >= min_af
        e = have[ab]
        return ok and ("%.2f %.2f %.2f" % (r.ani * 100, r.af_a * 100, r.af_b * 100)) == ("%.2f %.2f %.2f" % (e["ani"], e["af_a"], e["af_b"]))

    def check_rejected(ab):
        a, b = ab
        if not O.screen(gid[a], gid[b], screen / 100.0)[1]:
            return True
        r = O.pair(gid[a], gid[b])
        return r.ani < 0 or max(r.af_a, r.af_b) * 100 < min_af

    with ThreadPoolExecutor(threads) as ex:
        bad = sum(not x for x in ex.map(check_kept, kept)) + sum(not x for x in ex.map(check_rejected, rejected))
    return {"n_kept_checked": len(kept), "n_rejected_checked": len(rejected), "clades": len(clades), "mismatch": int(bad),
            "checked_against": "oracle.pair / oracle.screen on the same genomes, 2-decimal rows equal"}


def _write_clade_fasta(job):
    workload, c, per, outdir = job
    from skder_b200 import synth

    for m, contigs in enumerate(synth.clade_of(workload, c, per)):
        synth.write_fasta(os.path.join(outdir, "clade%03d_member%03d.fasta" % (c, m)), contigs, name="c%d_m%d" % (c, m))
    return per


def derep_wall(workload, mode, threads, n_clades=None):
    """`skder -d <mode>` -- the UNMODIFIED reference from baseline/_ref (tools/ref_runner.py) -- on the workload's genomes
    written as FASTA, with skder_b200/bin/skani first on PATH.  Returns a dict with wall seconds and the reference's own
    phase log; the FASTA files are generated and written before the clock starts."""
    from concurrent.futures import ProcessPoolExecutor

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import ref_runner

    if ref_runner.reference_tree() is None:
        return {"unavailable": "baseline/_ref not installed (tools/install_reference.py needs /root/reference once)"}
    nc, per, L = workload_shape(workload)
    nc = n_clades or nc
    need = nc * per * L * 1.02
    base = os.environ.get("SKB_BENCH_TMP")
    if not base:
        cands = [d for d in ("/dev/shm", tempfile.gettempdir()) if os.path.isdir(d) and shutil.disk_usage(d).free > 1.5 * need]
        if not cands:
            return {"unavailable": "no scratch space for %.0f GB of FASTA" % (need / 1e9)}
        base = cands[0]
    work = tempfile.mkdtemp(prefix="skb_derep_", dir=base)
    try:
        gdir = os.path.join(work, "genomes")
        os.makedirs(gdir)
        t0 = time.perf_counter()
        with ProcessPoolExecutor(min(threads, 32)) as ex:
            n = sum(ex.map(_write_clade_fasta, [(workload, c, per, gdir) for c in range(nc)]))
        t_write = time.perf_counter() - t0
        out = {"genomes": n, "fasta_dir": base, "fasta_gb": sum(os.path.getsize(os.path.join(gdir, f)) for f in os.listdir(gdir)) / 1e9,
               "setup_write_s": t_write, "threads": threads, "mode": mode,
               "command": "skder -g DIR -o OUT -d %s -c %d   (defaults: -i 99.5 -f 50)" % (mode, threads)}
        wall, reps, outdir = ref_runner.run_skder(gdir + "/", os.path.join(work, "out"), mode, SKDER_ANI, SKDER_AF, threads=threads,
                                                  env_extra={"SKB_PHASE_LOG": "1"}, timeout=3600)
        out.update({"wall_s": wall, "representatives": len(reps), "reference_phases_s": ref_runner.run_skder.last_phases})
        log = os.path.join(outdir, "Skani_Triangle_Edge_Output.txt.skani_b200.phases.json")
        if os.path.exists(log):
            out["shim_phases_s"] = json.load(open(log))
        return out
    except Exception as e:  # the throughput line must not be lost to a dereplication problem
        return {"error": "%s: %s" % (type(e).__name__, str(e)[-600:])}
    finally:
        shutil.rmtree(work, ignore_errors=True)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from skder_b200 import _lib, build, engine, multi, synth

    build.build()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torchrun --nproc-per-node %d" % (args.gpus, world, args.gpus))
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: bench.py has no CPU path for --impl ours")
    torch.cuda.set_device(local)
    numa_cpus = multi.bind_to_gpu_numa_node(torch, local) if world > 1 and os.environ.get("SKB_NO_NUMA_BIND") != "1" else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if args.workload in SEARCH_WORKLOADS:
        return run_ours_search(args, torch, dist, rank, world, local)

    nc, per, L = workload_shape(args.workload)
    n_full = nc * per
    pairs_full = n_full * (n_full - 1) // 2
    # every rank ingests its share of the clades (rank r: clades r, r+world, ...)
    from concurrent.futures import ThreadPoolExecutor

    t_gen = time.perf_counter()
    my_clades = list(range(rank, nc, world))
    packed = []

    def gen(c):
        return [engine.pack_contigs(g) for g in synth.clade_of(args.workload, c)]

    with ThreadPoolExecutor(max(1, min(32, (os.cpu_count() or 1) // max(world, 1)))) as ex:
        for clade in ex.map(gen, my_clades):
            packed += clade
    t_gen = time.perf_counter() - t_gen
    pin, views, keep, h2d_bytes = pinned_views(packed, torch)
    del packed
    arr = (C.POINTER(_lib.Packed) * len(views))(*[C.pointer(v) for v in views])
    # workload-wide genome number of every id after replication (rank-major order)
    canon = np.array([c * per + m for r in range(world) for c in range(r, nc, world) for m in range(per)], np.int64)

    eng = engine.Engine(local)
    L_ = eng._L
    phase_ms = []  # (add, replicate, index) wall ms of every sketch_all() call on this rank

    def sketch_all():
        """host packed genomes -> replicated, indexed sketch DB on every rank"""
        t0 = time.perf_counter()
        eng.clear()
        eng._ck(L_.skb_add_genomes(eng._h, len(views), arr), "skb_add_genomes")
        t1 = time.perf_counter()
        if world > 1:  # own genomes indexed first (repeat flags travel with the seeds); afterwards this rank owns their tables only
            multi.replicate_sketches(eng, dist, torch, sharded_index=True)
        t2 = time.perf_counter()
        eng.index()
        t3 = time.perf_counter()
        phase_ms.append(((t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3))
        if os.environ.get("SKB_BENCH_DEBUG") == "1" and rank == 0:
            sys.stderr.write("add %.2f ms  replicate %.2f ms  index %.2f ms\n" % phase_ms[-1])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    dbg = os.environ.get("SKB_BENCH_DEBUG") == "1"

    def triangle():
        t0 = time.perf_counter()
        if world == 1:
            edges, st = eng.triangle(GREEDY_SCREEN, GREEDY_MIN_AF)
            t1 = time.perf_counter()
        else:  # rows screened per rank, surviving pairs all-gathered, every pair evaluated by the owner of its reference
            _, st, st_screen = multi.triangle_sharded(eng, dist, torch, GREEDY_SCREEN, GREEDY_MIN_AF, to_host=False)
            st.ms_screen = st_screen.ms_screen
            t1 = time.perf_counter()
            edges = multi.gather_device_edges(eng, dist, torch, sort=False)
        if dbg and rank == 0:
            sys.stderr.write("triangle %.2f ms (screen %.2f ani %.2f) gather %.2f ms\n" % (
                (t1 - t0) * 1e3, st.ms_screen, st.ms_ani, (time.perf_counter() - t1) * 1e3))
        return edges, st

    # ---- warm-up (full e2e steps)
    for _ in range(args.warmup):
        sketch_all()
        triangle()
    # ---- e2e: host packed genomes -> edges on host, every step
    with ClockSampler(local) as clk_e2e:
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(args.steps):
            sketch_all()
            edges, st = triangle()
            d2h += edges.nbytes
        barrier()
        t_e2e = time.perf_counter() - t0
    # ---- index build alone, device-timed (reported beside `value`, which starts from the indexed sketch DB)
    eng.timer_start()
    eng.index()
    ms_index_dev = eng.timer_stop()
    # ---- value: sketches resident; device-timed on the library's stream
    l0 = eng.launches
    ms_ani, ms_screen, ms_anchor, n_anchor, st = [], [], [], [], None
    with ClockSampler(local) as clk:
        barrier()
        eng.timer_start()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            edges, st = triangle()
            ms_ani.append(st.ms_ani)
            ms_screen.append(st.ms_screen)
            ms_anchor.append(st.ms_anchor)
            n_anchor.append(st.n_anchor_launches)
        ms_dev = eng.timer_stop()
        barrier()
        t_wall = time.perf_counter() - t0
    launches = eng.launches - l0
    if world > 1:
        tt = torch.tensor([ms_dev, t_e2e, float(np.mean(ms_ani)), ms_index_dev], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_dev, t_e2e, ms_index_dev = float(tt[0]), float(tt[1]), float(tt[3])
        cnt = torch.tensor([st.n_pairs_screened, st.sum_query_seeds, st.sum_anchors, launches, h2d_bytes],
                           device="cuda", dtype=torch.int64)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        tot_screened, launches_all, h2d_all = int(cnt[0]), int(cnt[3]), int(cnt[4])
    else:
        tot_screened, launches_all, h2d_all = st.n_pairs_screened, launches, h2d_bytes
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:  # the edge list the last timed step returned
        dump_outputs(args.dump_outputs, "edges", canonical_table(edges, canon))

    ms_step = ms_dev / args.steps
    value = pairs_full / (ms_step / 1e3)
    e2e_value = pairs_full / (t_e2e / args.steps)
    # ---- roofline.  Algorithmic bytes per surviving pair for the whole pair stage = 32*S_q + 32*A + 20
    # (SURVEY.md section 8d / BASELINE.md section 4).  The dominant kernel is anchor_kernel; of the model's terms it
    # owns the query seed records (16*S_q), one index slot per probe (16*S_q) and the anchors written (16*A).
    # Duration = that kernel's average launch time from CUDA events the library records around every launch.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    stage_bytes = 32 * st.sum_query_seeds + 32 * st.sum_anchors + 20 * st.n_pairs_screened
    ani_ms = float(np.mean(ms_ani))
    stage_gbs = stage_bytes / (ani_ms / 1e3) / 1e9 if ani_ms > 0 else 0.0
    launches_per_step = max(1, int(np.mean(n_anchor)))
    anchor_ms = float(np.mean(ms_anchor)) / launches_per_step
    alg_bytes = (32 * st.sum_query_seeds + 16 * st.sum_anchors) / launches_per_step
    achieved = alg_bytes / (anchor_ms / 1e3) / 1e9 if anchor_ms > 0 else 0.0
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "anchor_kernel_traffic.json")))
        if tj.get("workload") == args.workload and world == 1:
            traffic = tj["dram_bytes_per_launch"]
    except Exception:
        pass
    threads = os.cpu_count() or 1
    line = {
        "metric": "genome pairs/sec ANI+AF", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64/int32 + f64", "data": "synthetic",
        "config": {"workload": workload_name(args.workload), "screen": GREEDY_SCREEN, "min_af": GREEDY_MIN_AF,
                   "pairs": pairs_full, "pairs_screened": tot_screened, "edges": int(len(edges)),
                   "l2": "inputs larger than L2 (sketch DB %.1f GB per rank)" % (
                       (st.sum_query_seeds and (n_full * L / 125 * 8 * 3) / 1e9) or 0.0),
                   "ms_screen": float(np.mean(ms_screen)), "ms_ani": ani_ms, "gen_s": t_gen,
                   "host_cpus_rank0": ("%d CPUs local to the GPU" % len(numa_cpus)) if numa_cpus else "unbound",
                   "wall_ms_per_step": t_wall / args.steps * 1e3,
                   # `value` starts from the indexed sketch DB (SURVEY 8d: "sketches resident on device"); the index
                   # build (seed tables + inverted marker index) is the prescreen's set-up and is reported here
                   "ms_index_device": ms_index_dev, "value_incl_index": pairs_full / ((ms_step + ms_index_dev) / 1e3)},
        "clocks": clk.summary(), "clocks_e2e": clk_e2e.summary(),
        "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h // args.steps,
                "ms_per_step": t_e2e / args.steps * 1e3,
                # rank 0's host-clock phases of the timed end-to-end steps (the rest of a step is skb_triangle + gather)
                "ms_upload_sketch": float(np.mean([p[0] for p in phase_ms[-args.steps:]])),
                "ms_replicate": float(np.mean([p[1] for p in phase_ms[-args.steps:]])),
                "ms_index": float(np.mean([p[2] for p in phase_ms[-args.steps:]]))},
        "gpu_launches": launches_all,
        "edges_sha256": canonical_edges(edges, canon),
        "roofline": {"bound": "hbm", "kernel": "anchor_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes": alg_bytes,
                     "ms_per_launch": anchor_ms, "launches_per_step": launches_per_step,
                     "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                     "note": "algorithmic (streaming-model) bytes over the kernel's time; the kernel is bound by the L1 data pipe "
                             "(one scattered 32-byte bucket read per lookup) and issue, its reference tables are L2-resident, "
                             "so real DRAM traffic (`traffic`) is far below the model; see DESIGN.md section 4"},
        "roofline_stage": {"kernels": "task_setup + anchor + chain + ends + finalize", "algorithmic_bytes": stage_bytes,
                           "ms": ani_ms, "achieved": stage_gbs, "unit": "GB/s", "frac": stage_gbs / peak},
    }
    # ---- outside the timed regions: oracle parity sample of the bench's own edge list, CPU baseline, dereplication
    if world == 1 and not args.no_parity:
        line["parity_sample"] = parity_sample(args.workload, edges, per, 12, 600, threads, GREEDY_SCREEN, GREEDY_MIN_AF)
    if world == 1 and not args.no_cpu:
        s_nc = min(nc, CPU_SAMPLE_CLADES)
        comp = cpu_triangle_components(args.workload, s_nc, CPU_SAMPLE_PER_CLADE, threads, GREEDY_SCREEN, GREEDY_MIN_AF)
        surv_full = nc * per * (per - 1) // 2
        v, t_full = cpu_extrapolate(comp, n_full, pairs_full, surv_full, with_sketch=False)
        line["cpu_baseline"] = {
            "value": v, "unit": "pairs/s", "cores": threads, "kind": "port",
            "sample": "INDICATIVE (oracle port, extrapolated): %d clades x %d members of %s (%d pairs, %d survivors): prescreen run "
                      "counting %.2fs, ANI/AF %.2fs on %d threads; sketches and the marker index resident (as for `value`); per-unit "
                      "costs scaled to the full workload.  `bench.py --impl reference` times the whole workload instead"
                      % (s_nc, CPU_SAMPLE_PER_CLADE, args.workload, comp["pairs"], comp["survivors"], comp["t_count"], comp["t_ani"],
                         threads)}
    if world == 1 and args.derep != "off":
        eng.close()  # the shim opens its own context on this GPU
        del pin
        line["derep"] = {m: derep_wall(args.workload, m, threads, n_clades=(10 if args.derep == "sample" else None))
                         for m in ("greedy", "dynamic")}
        if "wall_s" in line["derep"]["greedy"]:
            line["derep_wall_s"] = line["derep"]["greedy"]["wall_s"]
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_ours_search(args, torch, dist, rank, world, local):
    """config4: `skder -d low_mem_greedy` (reference src/skDER/skder.py:95-134) -- sketch the database once, then the
    greedy loop: in N50 order, every genome not yet accounted for is searched against the database.  SURVEY 8e: the
    database is sharded over the ranks (N/P genomes each, no replication); the rank that holds the query sketches it
    and broadcasts the sketch (seed records + marker keys, ~0.2 MB); every rank searches its shard; the hits' genome
    numbers are all-gathered into the accounted set.  The loop is sequential by construction."""
    from concurrent.futures import ThreadPoolExecutor

    from skder_b200 import _lib, engine, multi, synth

    nc, per, L = workload_shape(args.workload)
    nc = int(os.environ.get("SKB_SEARCH_CLADES", nc))  # bounded runs of the same shape
    n_full = nc * per
    t_gen = time.perf_counter()
    my_clades = list(range(rank, nc, world))

    def gen(c):
        return [engine.pack_contigs(g) for g in synth.clade_of(args.workload, c)]

    with ThreadPoolExecutor(max(1, min(32, (os.cpu_count() or 1) // max(world, 1)))) as ex:
        clades = list(ex.map(gen, my_clades))
    packed = [g for cl in clades for g in cl]
    my_ids = np.array([c * per + m for c in my_clades for m in range(per)], np.int64)  # workload-wide genome numbers
    local_of = {int(g): i for i, g in enumerate(my_ids)}
    t_gen = time.perf_counter() - t_gen
    n50 = np.zeros(n_full, np.int64)
    n50[my_ids] = [p.n50 for p in packed]
    if world > 1:
        t = torch.from_numpy(n50).cuda()
        dist.all_reduce(t)
        n50 = t.cpu().numpy()
    order = sorted(range(n_full), key=lambda g: (-int(n50[g]), g))
    pin, views, keep, h2d_bytes = pinned_views(packed, torch)
    arr = (C.POINTER(_lib.Packed) * len(views))(*[C.pointer(v) for v in views])
    eng = engine.Engine(local)
    eng_q = engine.Engine(local) if world > 1 else None  # scratch context: this rank's share of a batch of queries
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_run():
        """sketch + index the shard, then the greedy loop; returns (reps, pairs, t_sketch, t_loop, launches)"""
        l0 = eng.launches
        t0 = time.perf_counter()
        eng.clear()
        eng._ck(eng._L.skb_add_genomes(eng._h, len(views), arr), "skb_add_genomes")
        eng.index()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        n_db = eng.n_genomes
        all_db = np.arange(n_db, dtype=np.int32)
        accounted = np.zeros(n_full, bool)
        reps, rep_ids, hits = 0, [], []
        # The greedy loop is sequential, but a search result does not depend on the loop's state: the next K
        # candidates in N50 order that are not accounted for YET are searched in one call (one index_append, one
        # rectangle), and their results are applied in order -- a candidate an earlier one of the same batch accounts
        # for is skipped exactly as the sequential loop would skip it, its result discarded (SURVEY 8e: "speculation
        # cannot change the answer").  K adapts: it doubles while nothing is discarded and halves when something is.
        k_batch, pos, searched, wasted_all = 1, 0, 0, 0
        while pos < n_full:
            batch, p_ = [], pos
            while p_ < n_full and len(batch) < k_batch:
                if not accounted[order[p_]]:
                    batch.append(order[p_])
                p_ += 1
            pos = p_
            if not batch:
                break
            if world == 1:
                for g in batch:
                    eng.add([packed[local_of[g]]])
                ord_of_ctx, n_adds = np.arange(len(batch)), len(batch)
            else:
                # every rank sketches the candidates it holds into a scratch context; two small collectives bring all
                # of them to every rank (rank-major); ord_of_ctx maps a query's place in the context back to its place
                # in the batch (= N50 order)
                own = [j for j, g in enumerate(batch) if (g // per) % world == rank]
                eng_q.clear()
                if own:
                    eng_q.add([packed[local_of[batch[j]]] for j in own])
                _, n_adds = multi.append_gathered_sketches(eng_q, eng, dist, torch)
                ord_of_ctx = np.array([j for r in range(world) for j, g in enumerate(batch) if (g // per) % world == r], np.int64)
            try:
                eng.index_append()
                edges, st = eng.rect(all_db, list(range(n_db, n_db + len(batch))), screen=SEARCH_SCREEN, min_af=SEARCH_MIN_AF)
            finally:
                for _ in range(n_adds):
                    eng.pop_last_add()
            searched += len(batch)
            # skder.py:128: ANI >= cutoff and the AF in column 4 (the query's) >= cutoff, on the printed 2-decimal values
            hit = (np.round(edges["ani"], 2) >= SKDER_ANI) & (np.round(edges["af_b"], 2) >= SKDER_AF)
            qi = ord_of_ctx[edges["b"][hit].astype(np.int64) - n_db]
            ids = my_ids[edges["a"][hit]]
            if world > 1:  # one exchange per batch: (query ordinal << 32 | workload-wide genome number) of every hit
                rec = (qi << 32) | ids
                cnt = torch.tensor([len(rec)], device=dev, dtype=torch.int64)
                cnts = torch.zeros(world, device=dev, dtype=torch.int64)
                dist.all_gather_into_tensor(cnts, cnt)
                mx = max(int(cnts.max()), 1)
                send = torch.full((mx,), -1, device=dev, dtype=torch.int64)
                if len(rec):
                    send[: len(rec)] = torch.from_numpy(rec).to(dev)
                recv = torch.empty(world * mx, device=dev, dtype=torch.int64)
                dist.all_gather_into_tensor(recv, send)
                rec = recv[recv >= 0].cpu().numpy()
                qi, ids = rec >> 32, rec & 0xFFFFFFFF
            wasted, new_reps = 0, []
            for j, g in enumerate(batch):
                if accounted[g]:
                    wasted += 1
                    continue
                reps += 1
                rep_ids.append(g)
                new_reps.append(j)
                accounted[ids[qi == j]] = True
                accounted[g] = True
            wasted_all += wasted
            if keep_hits:  # this rank's rows of the searches whose results the loop used: (query, ref, ANI, AF ref, AF query)
                q_all = ord_of_ctx[edges["b"].astype(np.int64) - n_db]
                used = np.isin(q_all, new_reps)
                hits.append(np.stack([np.asarray(batch, np.float64)[q_all[used]], my_ids[edges["a"][used]].astype(np.float64),
                                      edges["ani"][used], edges["af_a"][used], edges["af_b"][used]], axis=1))
            k_batch = max(1, k_batch // 2) if wasted else min(SEARCH_BATCH_MAX, k_batch * 2)
        one_run.searched, one_run.wasted, one_run.rep_ids = searched, wasted_all, rep_ids
        one_run.hits = np.concatenate(hits) if hits else np.zeros((0, 5))
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        return reps, reps * n_full, t1 - t0, t2 - t1, eng.launches - l0

    keep_hits = bool(args.dump_outputs)
    for _ in range(min(args.warmup, 1)):
        one_run()
    res = []
    with ClockSampler(local) as clk:
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res.append(one_run())
        barrier()
        t_all = time.perf_counter() - t0
    if world > 1:
        tt = torch.tensor([t_all, float(np.mean([r[3] for r in res]))], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_all, t_loop = float(tt[0]), float(tt[1])
        ll = torch.tensor([res[-1][4]], device="cuda", dtype=torch.int64)
        dist.all_reduce(ll)
        launches_all = int(ll[0])
    else:
        t_loop, launches_all = float(np.mean([r[3] for r in res])), res[-1][4]
    if keep_hits and world > 1:
        shards = [None] * world
        dist.all_gather_object(shards, one_run.hits)
        one_run.hits = np.concatenate(shards)
    if rank == 0:
        if args.dump_outputs:  # what the last timed step selected, in selection order, and its searches' rows by (query, ref)
            used = dump_outputs(args.dump_outputs, "representatives", {"genome": one_run.rep_ids})
            h = one_run.hits[np.lexsort((one_run.hits[:, 1], one_run.hits[:, 0]))]
            dump_outputs(args.dump_outputs, "hits", {"query": h[:, 0], "ref": h[:, 1], "ani": h[:, 2], "af_ref": h[:, 3],
                                                     "af_query": h[:, 4]}, DUMP_MAX_BYTES - used)
        reps, pairs, t_sk, _, launches = res[-1]
        t_step = t_all / args.steps
        line = {
            "metric": "genome pairs/sec ANI+AF (search path)", "value": pairs / t_loop, "unit": "pairs/s",
            "n_gpus": world, "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": t_loop * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/int32 + f64", "data": "synthetic",
            "config": {"workload": workload_name(args.workload) if nc == workload_shape(args.workload)[0] else
                       "%s, first %d clades only (%d genomes)" % (workload_name(args.workload), nc, n_full),
                       "representatives": reps, "searches": reps, "pairs": pairs, "searches_per_s": reps / t_loop,
                       "ms_per_search": t_loop / reps * 1e3, "reps_sha256": ids_sha256(getattr(one_run, "rep_ids", [])),
                       "search_batching": "up to %d candidates per call, %d searched, %d results discarded (candidate "
                                          "accounted for by an earlier one of its batch)" % (
                                              SEARCH_BATCH_MAX, getattr(one_run, "searched", reps), getattr(one_run, "wasted", 0)), "ms_sketch_index_db": float(np.mean([r[2] for r in res])) * 1e3,
                       "gen_s": t_gen,
                       "timing": "host clock between device synchronisations, max over ranks: the loop is sequential host "
                                 "logic around ~%d small launches per search" % max(1, launches // max(reps, 1)),
                       "sharding": "database sharded N/P per rank; a batch's queries are sketched by the ranks that hold them, "
                                   "their sketches all-gathered (two collectives per batch); hit ids all-gathered" if world > 1
                                   else "one GPU holds the database"},
            "clocks": clk.summary(),
            "e2e": {"value": pairs / t_step, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d_bytes) * world + reps * int(L // 4),
                    "d2h_bytes_per_step": int(32 * per * reps), "ms_per_step": t_step * 1e3,
                    "note": "database upload + sketch + index + the whole search loop (queries uploaded one by one)"},
            "gpu_launches": int(launches_all * args.steps),
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", default="config3", choices=["tiny", "tinyr", "tiny4", "config2", "config3", "config3r", "config4", "config5"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity sample")
    ap.add_argument("--derep", choices=["off", "sample", "full"], default=os.environ.get("SKB_BENCH_DEREP", "full"),
                    help="dereplication wall time through the unmodified reference (N=1): whole workload, 10 clades, or skip")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float64): the edge list "
                         "sorted by genome number (edges_a, edges_b, edges_ani, edges_af_a, edges_af_b) or, for the search "
                         "workloads, the representatives in selection order and the rows of their searches sorted by (query, "
                         "ref) (hits_query, hits_ref, hits_ani, hits_af_ref, hits_af_query); a seeded row sample above 64 MB")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
