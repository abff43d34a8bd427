"""Multi-GPU plumbing (one process per GPU, torch.distributed): sketch replication and edge gather.

The pair triangle shards by rows with no data-path collective (skb_triangle's part/n_parts); the
only exchanges are (1) replicating the sketches every rank made from its share of the genomes --
one padded NCCL all-gather per array straight out of / into the library's device buffers -- and
(2) gathering the sparse edge lists to rank 0.
"""
import ctypes as C

import numpy as np

from .engine import EDGE_DTYPE


class _DevArray:
    """Zero-copy torch view of library-owned device memory via __cuda_array_interface__."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i8", "data": (int(ptr), False), "version": 2}


def _dev_tensor(torch, ptr, n, device):
    if n == 0 or not ptr:
        return torch.empty(0, dtype=torch.int64, device=device)
    return torch.as_tensor(_DevArray(ptr, n), device=device)


def replicate_sketches(eng, dist, torch, sharded_index=False):
    """Every rank holds the sketches of its own genomes; afterwards every rank holds all of them,
    ordered by (rank, local order).  Collective: all ranks must call.

    sharded_index: the rank first builds the seed tables of its own genomes (their repeat flags are part of the seed
    records and travel with them), keeps the tables across the exchange, and afterwards owns exactly those genomes
    (skb_set_owned): the next Engine.index() reuses the tables and adds only the chunk tables and the marker index of
    the whole set -- 1/P of the table work and memory per rank, done once -- and triangle_sharded() sends every pair to
    the rank that owns its reference genome."""
    import os
    import sys
    import time

    prof = os.environ.get("SKB_REPL_PROFILE") == "1"
    tm = [time.perf_counter()]

    def lap():
        if prof:
            torch.cuda.synchronize()
            tm.append(time.perf_counter())

    world, rank = dist.get_world_size(), dist.get_rank()
    if sharded_index and eng.n_genomes:
        eng.index_seed_tables()
    lap()
    metas, gathered = _allgather_sketches(eng, dist, torch, lap)
    eng.clear(keep_tables=sharded_index)
    _import_gathered(eng, metas, gathered, keep_flags=sharded_index)
    if sharded_index:
        eng.set_owned(sum(int(m["n"]) for m in metas[:rank]), int(metas[rank]["n"]))
    lap()
    if prof and rank == 0:
        sys.stderr.write("replicate: own index %.2f  meta %.2f  all-gather %.2f  import %.2f ms\n" % tuple(
            (b - a) * 1e3 for a, b in zip(tm, tm[1:])))
    return metas


def _allgather_sketches(eng, dist, torch, lap=lambda: None):
    """Raw sketches (seed records, marker keys) and host tables of every rank's context, all-gathered: returns
    (metas per rank, [(seeds, stride), (marker keys, stride)] as padded device tensors)."""
    device = torch.device("cuda", eng.device)
    v = eng.sketch_view()
    n = v.n_genomes
    nctg = int(v.n_contigs)
    meta = {  # an empty context (a rank without queries in this batch) has null host tables
        "n": n, "n_seeds": v.n_seeds, "n_mkeys": v.n_marker_keys, "marker_c": eng.marker_compression,
        "seed_off": np.ctypeslib.as_array(v.host_seed_off, shape=(n + 1,)).copy() if n else np.zeros(1, np.uint64),
        "total_len": np.ctypeslib.as_array(v.host_total_len, shape=(n,)).copy() if n else np.zeros(0, np.uint64),
        "ctg_off": np.ctypeslib.as_array(v.host_ctg_off, shape=(n + 1,)).copy() if n else np.zeros(1, np.uint32),
        "ctg_len": np.ctypeslib.as_array(v.host_ctg_len, shape=(nctg,)).copy() if nctg else np.zeros(0, np.uint32),
    }
    metas = _exchange_meta(meta, dist, torch, device if dist.get_backend() == "nccl" else None)
    lap()
    world = dist.get_world_size()
    gathered = []
    for key, ptr, cnt in (("n_seeds", v.dev_seeds, v.n_seeds), ("n_mkeys", v.dev_marker_keys, v.n_marker_keys)):
        mx = max(int(m[key]) for m in metas)
        send = torch.zeros(max(mx, 1), dtype=torch.int64, device=device)
        if cnt:
            send[:cnt].copy_(_dev_tensor(torch, ptr, cnt, device))
        recv = torch.empty(world * max(mx, 1), dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(recv, send)
        gathered.append((recv, max(mx, 1)))
    torch.cuda.synchronize(device)
    lap()
    return metas, gathered


def _import_gathered(eng, metas, gathered, keep_flags=False):
    """Append every rank's gathered sketches to `eng`, rank-major; returns the number of import (= add) calls made."""
    (seeds, s_stride), (mkeys, m_stride) = gathered
    if metas and metas[0]["marker_c"] != eng.marker_compression:  # the sketch view does not carry it (skb_import_sketches)
        raise ValueError("sketches made at marker compression %d cannot join a context at %d"
                         % (metas[0]["marker_c"], eng.marker_compression))
    calls = 0
    for r, m in enumerate(metas):
        if m["n"] == 0:
            continue
        so = np.ascontiguousarray(m["seed_off"], np.uint64)
        tl = np.ascontiguousarray(m["total_len"], np.uint64)
        co = np.ascontiguousarray(m["ctg_off"], np.uint32)
        cl = np.ascontiguousarray(m["ctg_len"], np.uint32)
        eng._ck(
            eng._L.skb_import_sketches(
                eng._h, int(m["n"]), C.c_void_p(seeds.data_ptr() + 8 * r * s_stride), int(m["n_seeds"]),
                C.c_void_p(mkeys.data_ptr() + 8 * r * m_stride), int(m["n_mkeys"]), so.ctypes.data, tl.ctypes.data,
                co.ctypes.data, cl.ctypes.data, 1 if keep_flags else 0),
            "skb_import_sketches",
        )
        calls += 1
    return calls


def append_gathered_sketches(src, dst, dist, torch):
    """Search path: every rank sketched its share of a batch of query genomes into the scratch context `src`; all of
    them are appended to `dst` on every rank, rank-major (two small collectives per batch instead of two broadcasts per
    query).  Returns (metas per rank, number of add calls to pop afterwards).  Collective: all ranks must call."""
    metas, gathered = _allgather_sketches(src, dist, torch)
    return metas, _import_gathered(dst, metas, gathered, keep_flags=False)


def _exchange_meta(meta, dist, torch, device):
    """The per-rank host tables of replicate_sketches as two tensor all-gathers (sizes, then one padded int64 blob)
    instead of pickled objects: no Python object serialisation in the per-step path.  Every rank must have sketched at
    the same marker compression (the screen compares marker counts across genomes): ValueError on every rank if not."""
    world = dist.get_world_size()
    n, nctg = int(meta["n"]), len(meta["ctg_len"])
    mc = int(meta.get("marker_c", 1000))  # tables without it were sketched at skani's default
    head = torch.tensor([n, int(meta["n_seeds"]), int(meta["n_mkeys"]), nctg, mc], dtype=torch.int64, device=device)
    heads = torch.zeros(world * 5, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(heads, head)
    heads = heads.cpu().numpy().reshape(world, 5)
    if len(set(heads[:, 4].tolist())) > 1:
        raise ValueError("ranks sketched at different marker compressions (-m): %s" % heads[:, 4].tolist())
    size = lambda h: (int(h[0]) + 1) + int(h[0]) + (int(h[0]) + 1) + int(h[3])
    mx = max(1, max(size(h) for h in heads))
    blob = np.zeros(mx, np.int64)
    parts = [np.asarray(meta["seed_off"], np.uint64).view(np.int64), np.asarray(meta["total_len"], np.uint64).view(np.int64),
             np.asarray(meta["ctg_off"], np.int64), np.asarray(meta["ctg_len"], np.int64)]
    cat = np.concatenate(parts) if parts else np.zeros(0, np.int64)
    blob[: len(cat)] = cat
    send = torch.from_numpy(blob).to(device) if device is not None else torch.from_numpy(blob)
    recv = torch.zeros(world * mx, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(recv, send)
    recv = recv.cpu().numpy().reshape(world, mx)
    out = []
    for r in range(world):
        n_r, ns, nm, nc, mc = (int(x) for x in heads[r])
        o = 0
        seed_off = recv[r, o:o + n_r + 1].view(np.uint64).copy(); o += n_r + 1
        total_len = recv[r, o:o + n_r].view(np.uint64).copy(); o += n_r
        ctg_off = recv[r, o:o + n_r + 1].astype(np.uint32); o += n_r + 1
        ctg_len = recv[r, o:o + nc].astype(np.uint32)
        out.append({"n": n_r, "n_seeds": ns, "n_mkeys": nm, "marker_c": mc, "seed_off": seed_off, "total_len": total_len,
                    "ctg_off": ctg_off, "ctg_len": ctg_len})
    return out


def triangle_sharded(eng, dist, torch, screen, min_af, to_host=False):
    """The triangle over P ranks, sharded by reference genome (after replicate_sketches(sharded_index=True) + index()):
    every rank screens its rows, the surviving pair lists (8 bytes per pair) are all-gathered over NCCL, and every rank
    evaluates the pairs whose reference genome it owns.  Returns (edges or None, stats of the pair stage, stats of the
    screen); edges are this rank's, sorted by the gathered pair order."""
    world, rank = dist.get_world_size(), dist.get_rank()
    device = torch.device("cuda", eng.device)
    ptr, n, st_screen = eng.screen_triangle(screen, part=rank, n_parts=world)
    counts = torch.zeros(world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(counts, torch.tensor([n], dtype=torch.int64, device=device))
    counts = counts.tolist()
    mx = max(max(counts), 1)
    send = torch.zeros(mx, dtype=torch.int64, device=device)
    if n:
        send[:n].copy_(_dev_tensor(torch, ptr, n, device))
    recv = torch.empty(world * mx, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(recv, send)
    allp = torch.cat([recv[r * mx: r * mx + c] for r, c in enumerate(counts)]) if sum(counts) else recv[:0]
    torch.cuda.current_stream(device).synchronize()  # the library reads the list on its own stream
    edges, st = eng.pairs_edges(allp.data_ptr(), int(allp.numel()), owned_only=True, min_af=min_af, to_host=to_host)
    return edges, st, st_screen


def gather_edges(edges, dist, torch, device=None, sort=True):
    """Variable-length edge arrays of all ranks -> one array on rank 0 (empty elsewhere), sorted by (a, b) if
    `sort` (each rank's part is already sorted, so rank-major order is deterministic too; skDER's consumers do
    not depend on row order, SURVEY section 4 fact 4).
    Two small collectives: the counts, then one padded gather of the raw 32-byte records."""
    world, rank = dist.get_world_size(), dist.get_rank()
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    counts = torch.zeros(world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(counts, torch.tensor([len(edges)], dtype=torch.int64, device=device))
    counts = counts.tolist()
    mx = max(max(counts), 1)
    send = torch.zeros(mx * EDGE_DTYPE.itemsize, dtype=torch.uint8, device=device)
    if len(edges):
        send[: len(edges) * EDGE_DTYPE.itemsize].copy_(torch.from_numpy(np.ascontiguousarray(edges).view(np.uint8)))
    recv = torch.empty(world * mx * EDGE_DTYPE.itemsize, dtype=torch.uint8, device=device) if rank == 0 else None
    dist.gather(send, list(recv.chunk(world)) if rank == 0 else None, dst=0)
    return _finish_gather(recv, counts, mx, world, rank, sort)


_pinned = {}


def _to_host(t):
    """Device tensor -> numpy through a cached pinned buffer (a pageable .cpu() of a few MB costs ~2 ms)."""
    if t.device.type != "cuda":
        return t.numpy()
    import torch

    buf = _pinned.get("buf")
    if buf is None or buf.numel() < t.numel():
        buf = torch.empty(max(t.numel(), 1 << 22), dtype=torch.uint8).pin_memory()
        _pinned["buf"] = buf
    view = buf[: t.numel()]
    view.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return view.numpy()


def _finish_gather(recv, counts, mx, world, rank, sort):
    if rank != 0:
        return np.zeros(0, EDGE_DTYPE)
    # byte slices, not structured ones: numpy copies structured arrays field by field (1.8 ms for 122,500 records)
    sz = EDGE_DTYPE.itemsize
    flat = _to_host(recv).view(np.uint8).reshape(world, mx * sz)
    out = np.concatenate([flat[r, : c * sz] for r, c in enumerate(counts)]).view(EDGE_DTYPE)  # a copy: the buffer is reused
    if not sort:
        return out
    key = (out["a"].astype(np.uint64) << np.uint64(32)) | out["b"].astype(np.uint64)
    return out[np.argsort(key, kind="stable")]


def gather_device_edges(eng, dist, torch, sort=True):
    """gather_edges for a result that is still on the device (Engine.triangle(to_host=False)): the per-rank lists go
    from the library's buffer over NCCL to rank 0 and reach host memory once, there."""
    import os
    import sys
    import time

    prof = os.environ.get("SKB_GATHER_PROFILE") == "1"
    tm = [time.perf_counter()]

    def lap():
        if prof:
            torch.cuda.synchronize()
            tm.append(time.perf_counter())

    world, rank = dist.get_world_size(), dist.get_rank()
    device = torch.device("cuda", eng.device)
    ptr, n = eng.device_edges()
    counts = torch.zeros(world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(counts, torch.tensor([n], dtype=torch.int64, device=device))
    counts = counts.tolist()
    lap()
    mx = max(max(counts), 1)
    words = EDGE_DTYPE.itemsize // 8
    send = torch.empty(mx * words, dtype=torch.int64, device=device)
    if n:
        send[: n * words].copy_(_dev_tensor(torch, ptr, n * words, device))
    recv = torch.empty(world * mx * words, dtype=torch.int64, device=device) if rank == 0 else None
    lap()
    dist.gather(send, list(recv.chunk(world)) if rank == 0 else None, dst=0)
    lap()
    out = _finish_gather(recv.view(torch.uint8) if rank == 0 else None, counts, mx, world, rank, sort)
    lap()
    if prof and rank == 0:
        sys.stderr.write("gather: counts %.2f  stage %.2f  gather %.2f  to-host %.2f ms\n" % tuple(
            (b - a) * 1e3 for a, b in zip(tm, tm[1:])))
    return out


def partition_rows(n, part, n_parts):
    """Rows of the pair triangle owned by `part`, and how many pairs that is.  Rows are dealt in zig-zag order
    (0..P-1, P-1..0, ...) so that all parts hold the same number of pairs (row a has n-1-a); the same rule as
    row_owner() in csrc/skb_common.cuh."""
    a = np.arange(n)
    m = a % (2 * n_parts)
    rows = a[np.where(m < n_parts, m, 2 * n_parts - 1 - m) == part]
    return rows, int((n - 1 - rows).sum())


def bind_to_gpu_numa_node(torch, device_index):
    """Pin this process (and so its first-touch page placement) to the CPUs local to its GPU's PCIe root before any
    pinned staging buffer is allocated.  With one process per GPU and no binding, the pinned buffers of all ranks tend
    to land on whichever socket the launcher ran on and every upload of the far GPUs crosses the socket interconnect:
    eight simultaneous uploads then share ~170 GB/s instead of running at ~50 GB/s each.  Returns the CPU list used,
    or None where sysfs does not say (single-socket boxes, containers without /sys/bus/pci)."""
    import os

    try:
        bdf = torch.cuda.get_device_properties(device_index).pci_bus_id if hasattr(
            torch.cuda.get_device_properties(device_index), "pci_bus_id") else None
        if not bdf:
            import pynvml

            pynvml.nvmlInit()
            vis = [x for x in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if x.strip()]
            phys = int(vis[device_index]) if vis and vis[device_index].strip().isdigit() else device_index
            bdf = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
            bdf = bdf.decode() if isinstance(bdf, bytes) else bdf
        bdf = bdf.lower()
        if len(bdf.split(":")[0]) == 8:  # NVML prints a 32-bit domain, sysfs a 16-bit one
            bdf = bdf[4:]
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bdf
        cpus = set()
        for part in open(path).read().strip().split(","):
            if not part:
                continue
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus or cpus == allowed:
            return None
        os.sched_setaffinity(0, cpus)
        return sorted(cpus)
    except Exception:
        return None

