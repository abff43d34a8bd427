// Shared definitions for the sm_100a ANI/AF kernels: record layouts, device views, small helpers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/skani_b200.h"

namespace skb {

// ---- fixed algorithm constants (skani defaults; see DESIGN.md section 3) ----------------------
constexpr int K_SEED = 15;
constexpr int K_MARKER = 21;
constexpr uint64_t C_SEED = 125;
constexpr uint64_t C_MARKER = 1000;  // skani's -m default; a context's value is skb_set_marker_compression's
constexpr uint64_t THR_SEED = 0xFFFFFFFFFFFFFFFFull / C_SEED;
// markers are kept iff mm_hash64 < marker_threshold(m) (SketchBatch::thr_marker)
__host__ __device__ inline uint64_t marker_threshold(uint64_t m) { return 0xFFFFFFFFFFFFFFFFull / m; }
constexpr uint64_t MASK_MARKER = (~0ull) >> (64 - 2 * K_MARKER);
constexpr uint64_t MASK_SEED = (~0ull) >> (64 - 2 * K_SEED);
constexpr uint32_t CONTIG_PAD = 4096;  // virtual gap between contigs in genome coordinates

// ---- packed seed record: kmer(30) << 34 | padded_pos(32) << 2 | rep << 1 | strand -------------
__host__ __device__ inline uint32_t seed_kmer(uint64_t s) { return (uint32_t)(s >> 34); }
__host__ __device__ inline uint32_t seed_pos(uint64_t s) { return (uint32_t)((s >> 2) & 0xffffffffu); }
__host__ __device__ inline int seed_rep(uint64_t s) { return (int)((s >> 1) & 1); }
__host__ __device__ inline int seed_strand(uint64_t s) { return (int)(s & 1); }

// ---- marker key of the inverted index: marker(42) << 22 | genome id(22) -----------------------
constexpr int GID_BITS = 22;
constexpr uint64_t GID_MASK = (1ull << GID_BITS) - 1;

constexpr uint64_t TAB_EMPTY = 0xFFFFFFFFFFFFFFFFull;

// minimap2/skani invertible 64-bit mix; first line is ~(key + (key << 21)) (see oracle).  The shift-add
// steps are written as the multiplications they are (x + (x<<3) + (x<<8) = 265 x, ...): identical mod
// 2^64, but they issue on the FMA pipe (IMAD) instead of piling 64-bit shifts/adds on the ALU pipe,
// which is what bounded the sketch kernel (ncu: 39% math-pipe throttle).
__host__ __device__ inline uint64_t mm_hash64(uint64_t key) {
    key = ~(key * 0x200001ull);
    key = key ^ (key >> 24);
    key = key * 265ull;
    key = key ^ (key >> 14);
    key = key * 21ull;
    key = key ^ (key >> 28);
    key = key * 0x80000001ull;
    return key;
}

// Rows of the pair triangle are dealt to partitions in zig-zag order (0..P-1, P-1..0, 0..P-1, ...).  Row a holds
// n-1-a pairs, so every two consecutive rounds give all partitions the same number of pairs (a plain round-robin
// leaves partition 0 with 4% more pairs than partition P-1 at n = 5000, P = 4).
__host__ __device__ inline uint32_t row_owner(uint32_t a, uint32_t P) {
    const uint32_t m = a % (2 * P);
    return m < P ? m : 2 * P - 1 - m;
}
__host__ __device__ inline uint32_t row_local(uint32_t a, uint32_t P) { return 2 * (a / (2 * P)) + (a % (2 * P) >= P ? 1u : 0u); }
__host__ __device__ inline uint32_t row_global(uint32_t rl, uint32_t part, uint32_t P) {
    return (rl >> 1) * 2 * P + ((rl & 1) ? 2 * P - 1 - part : part);
}
__host__ __device__ inline uint32_t rows_owned(uint32_t n, uint32_t part, uint32_t P) {
    const uint32_t rem = n % (2 * P);
    return 2 * (n / (2 * P)) + (rem > part ? 1u : 0u) + (rem > 2 * P - 1 - part ? 1u : 0u);
}

// Seed index layout: buckets of 4 slots (one 32-byte sector), one home bucket per k-mer, overflow into the
// following buckets behind a per-bucket flag (skb_probe.cuh).
constexpr uint32_t BUCKET = 4;

// Per-task scratch slabs of the pair stage (anchors: u64, DP results: u32): SLAB entries per task, contiguous.
// (Round 2 tried interleaving the slabs of the 32 tasks a chain_kernel warp holds, in pieces of 4 entries, so that its
// loads touch 8 lines instead of 32: chain_kernel did not move -- it is not bound by its loads -- and anchor_kernel,
// whose warp-wide anchor stores then touch 8 lines instead of 2, went from 5.0 to 5.4 ms per batch.)
constexpr int SLAB = 256;  // entries per task (= MAXA, skb_ani.cuh)
__host__ __device__ inline size_t slab_base(uint32_t t) { return (size_t)t * SLAB; }
__host__ __device__ inline uint32_t slab_off(uint32_t i) { return i; }
__host__ __device__ inline size_t slab_entries(uint64_t tasks) { return (size_t)tasks * SLAB; }

// Device view of the sketch DB (all pointers device memory)
struct DbView {
    int32_t n_genomes;
    const uint64_t *seeds;       // position-ordered records, all genomes
    const uint64_t *g_seed_off;  // [n+1]
    const uint64_t *tab;         // open-addressing seed index, all genomes
    const uint64_t *g_tab_off;   // [n+1]
    const uint32_t *g_tab_buckets; // [n] buckets per table (seeds x 2, 1 or 1/2: skb_index), 4 slots each
    const uint32_t *chunk_begin; // genome g: n_chunks(g)+1 entries at g_chunk_off[g] + g (seed index relative to genome)
    const uint32_t *chunk_start; // [total chunks] padded coordinate of first base
    const uint32_t *chunk_len;   // [total chunks]
    const uint32_t *g_chunk_off; // [n+1]
    const uint32_t *ctg_pstart;  // [total contigs] padded coordinate of contig base 0
    const uint32_t *ctg_len;     // [total contigs]
    const uint32_t *g_ctg_off;   // [n+1]
    const uint64_t *g_total_len; // [n]
    const uint64_t *markers;     // per-genome sorted unique markers
    const uint64_t *g_marker_off;// [n+1]
    const uint64_t *inv_keys;    // sorted unique (marker << 22 | gid)
    int64_t n_inv;
};

struct PairOut {
    double ani, ani_raw, af_q, af_r;
    int64_t n_anchors, n_seeds, span_q, span_r;
    int32_t n_chains, swapped;
};

}  // namespace skb
