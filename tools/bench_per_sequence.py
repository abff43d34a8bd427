"""skani's per-sequence mode (-i; DESIGN.md section 3) on a plasmid/virus-like workload on one GPU.

  python tools/bench_per_sequence.py [--files 200] [--records 1000] [--out result.json]

Workload (seeded): 200 multi-FASTA files x 1,000 records of 1-20 kb (~2.1 Gbp, 200 k sequences).  The records form
10,000 clades of 20 members, 0.05-0.5 % apart, dealt round-robin over the files, so that about 1.9 M within-clade pairs
can pass the screen at -m 200.  Reported, with the card's name and power limit read in the same run:
- the sketch stage's device time (CUDA events on the context's stream around the add call, upload included) of
  skb_add_sequences on the packed files, against the same records added as separate genomes (skb_pack_contigs +
  skb_add_genomes), alternated over --rounds; the two sketch databases are asserted identical (seed and marker arrays on
  the device, offsets and contig tables on the host);
- `triangle -i` at -m 200 on the per-sequence context: skb_stats' screen and pair-stage device times, pairs screened
  and edges.  The screen's count matrix is dense (N^2 cells); if the device cannot hold it, the error is reported.
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
from bench_estimators import card  # noqa: E402

SEED = 20261024


def workload(files, records, clades, tmp):
    """write the FASTA files; returns (paths, the records' sequences as bytes in (file, record) order)"""
    rng = np.random.default_rng(SEED)
    lens = rng.integers(1000, 20001, clades)
    anc = [rng.integers(0, 4, int(n), dtype=np.uint8) for n in lens]
    acgt = np.frombuffer(b"ACGT", np.uint8)
    paths, seqs = [], []
    for f in range(files):
        p = os.path.join(tmp, "f%03d.fa" % f)
        with open(p, "wb") as out:
            for r in range(records):
                c = (f * records + r) % clades
                g = anc[c].copy()
                k = rng.binomial(len(g), rng.uniform(0.0005, 0.005))
                pos = rng.integers(0, len(g), k)
                g[pos] = (g[pos] + rng.integers(1, 4, k).astype(np.uint8)) & 3
                s = acgt[g].tobytes()
                seqs.append(s)
                out.write(b">f%03d_r%04d clade %d\n" % (f, r, c))
                out.write(b"\n".join(s[i:i + 80] for i in range(0, len(s), 80)) + b"\n")
        paths.append(p)
    return paths, seqs


def device_array(ptr, n):
    import torch

    class View:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i8", "data": (int(ptr), False), "version": 2}

    return torch.as_tensor(View(), device="cuda")


def same_sketch_db(ea, eb):
    import torch

    va, vb = ea.sketch_view(), eb.sketch_view()
    n = va.n_genomes
    assert n == vb.n_genomes and va.n_seeds == vb.n_seeds and va.n_marker_keys == vb.n_marker_keys
    for f, k in (("host_seed_off", n + 1), ("host_total_len", n), ("host_ctg_off", n + 1), ("host_ctg_len", va.n_contigs)):
        assert np.array_equal(np.ctypeslib.as_array(getattr(va, f), (k,)), np.ctypeslib.as_array(getattr(vb, f), (k,))), f
    for f, k in (("dev_seeds", va.n_seeds), ("dev_marker_keys", va.n_marker_keys)):
        assert torch.equal(device_array(getattr(va, f), k), device_array(getattr(vb, f), k)), f
    torch.cuda.synchronize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=200)
    ap.add_argument("--records", type=int, default=1000)
    ap.add_argument("--clades", type=int, default=10000)
    ap.add_argument("--m", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out")
    a = ap.parse_args()
    from skder_b200 import engine

    res = {"card": card(0), "files": a.files, "records": a.records, "clades": a.clades, "m": a.m}
    with tempfile.TemporaryDirectory(prefix="bench_per_seq.") as tmp:
        t0 = time.time()
        paths, seqs = workload(a.files, a.records, a.clades, tmp)
        res["gen_s"] = round(time.time() - t0, 1)
        res["bases"] = int(sum(len(s) for s in seqs))
        t0 = time.time()
        packed = engine.pack_fasta_many(paths, threads=os.cpu_count())
        res["pack_files_s"] = round(time.time() - t0, 2)
        t0 = time.time()
        single = [engine.pack_contigs([s]) for s in seqs]
        res["pack_records_s"] = round(time.time() - t0, 2)
        del seqs
        ea, eb = engine.Engine(0), engine.Engine(0)
        for e in (ea, eb):
            e.set_marker_compression(a.m)
        ms_seq, ms_sep = [], []
        for r in range(a.rounds + 1):  # round 0 warms both paths up
            for e, add, ms in ((ea, lambda: ea.add(packed, per_sequence=True), ms_seq), (eb, lambda: eb.add(single), ms_sep)):
                e.clear()
                e.timer_start()
                add()
                t = e.timer_stop()
                if r:
                    ms.append(round(t, 2))
        same_sketch_db(ea, eb)
        res["sketch_ms_per_sequence"], res["sketch_ms_separate"] = ms_seq, ms_sep
        res["genomes"] = ea.n_genomes
        eb.close()
        del single
        t0 = time.time()
        ea.index()
        res["index_s"] = round(time.time() - t0, 2)
        try:
            edges, st = ea.triangle(screen=80.0, min_af=15.0)
            res["triangle"] = {"ms_screen": round(st.ms_screen, 1), "ms_ani": round(st.ms_ani, 1),
                               "ms_total": round(st.ms_total, 1), "pairs_total": st.n_pairs_total,
                               "pairs_screened": st.n_pairs_screened, "edges": st.n_edges}
        except Exception as ex:  # the dense screen matrix at this N is what this run is meant to show
            res["triangle"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        ea.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
