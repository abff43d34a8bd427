// On-demand seed tables (skb_api.cu, DESIGN.md section 2): when the tables of every genome do not fit the table
// budget, an edge call builds the tables of the genomes that are the reference of a surviving pair, a block of them
// at a time, evaluates that block's pairs, and merges the blocks' edges back into the order of the call's pair list, the
// order the resident path leaves.
//
// A block is a list of genome ids, ascending.  Its tables are laid out back to back from slot 0 of the table buffer;
// block_layout_kernel writes their offsets and bucket counts into the per-genome arrays DbView reads, so the pair-stage
// kernels read a block exactly as they read resident tables.
#pragma once
#include "skb_common.cuh"
#include "skb_probe.cuh"

namespace skb {

// mark[r] = 1 for the reference genome r of every pair (the one with more seeds; ties: b -- pair_setup_kernel's rule)
__global__ void ref_mark_kernel(const uint64_t *__restrict__ g_seed_off, const unsigned long long *__restrict__ pairs,
                                int64_t n_pairs, uint32_t n_genomes, uint8_t *__restrict__ mark) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs) return;
    const uint32_t a = (uint32_t)(pairs[t] >> 32), b = (uint32_t)(pairs[t] & 0xffffffffu);
    if (a >= n_genomes || b >= n_genomes) return;
    const uint64_t nsa = g_seed_off[a + 1] - g_seed_off[a], nsb = g_seed_off[b + 1] - g_seed_off[b];
    mark[nsb < nsa ? a : b] = 1;
}

// the block's k genomes gid[j]: table offset loc_off[j] (in words of the table buffer) and nb[j] buckets
__global__ void block_layout_kernel(const uint32_t *__restrict__ gid, const uint64_t *__restrict__ loc_off,
                                    const uint32_t *__restrict__ nb, int k, uint64_t *__restrict__ g_tab_off,
                                    uint32_t *__restrict__ g_tab_buckets) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    g_tab_off[gid[j]] = loc_off[j];
    g_tab_buckets[gid[j]] = nb[j];
}

// thread t of the block's seed records: pref[j] .. pref[j + 1] are genome gid[j]'s (pref[k] in all); its global index
__device__ __forceinline__ bool block_seed(const uint64_t *__restrict__ g_seed_off, const uint32_t *__restrict__ gid,
                                           const uint64_t *__restrict__ pref, int k, uint64_t t, uint32_t &g, uint64_t &i) {
    const uint64_t total = pref[k];
    const int j = genome_of_warp(pref, k, t < total ? t : total - 1);  // all 32 lanes
    if (t >= total) return false;
    g = gid[j];
    i = g_seed_off[g] + (t - pref[j]);
    return true;
}

// tab_insert_kernel over the seed records of the block's genomes
__global__ void block_tab_insert_kernel(const uint64_t *__restrict__ seeds, const uint64_t *__restrict__ g_seed_off,
                                        const uint32_t *__restrict__ gid, const uint64_t *__restrict__ pref, int k,
                                        uint64_t *tab, const uint64_t *__restrict__ g_tab_off,
                                        const uint32_t *__restrict__ g_tab_buckets) {
    uint32_t g;
    uint64_t i;
    if (!block_seed(g_seed_off, gid, pref, k, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, g, i)) return;
    tab_insert_rec(reinterpret_cast<unsigned long long *>(tab + g_tab_off[g]), g_tab_buckets[g], seeds[i] | 2ull);
}

// rep_flag_kernel over the seed records of the block's genomes
__global__ void block_rep_flag_kernel(uint64_t *seeds, const uint64_t *__restrict__ g_seed_off,
                                      const uint32_t *__restrict__ gid, const uint64_t *__restrict__ pref, int k,
                                      uint64_t *tab, const uint64_t *__restrict__ g_tab_off,
                                      const uint32_t *__restrict__ g_tab_buckets, int max_mult) {
    uint32_t g;
    uint64_t i;
    if (!block_seed(g_seed_off, gid, pref, k, (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, g, i)) return;
    const uint64_t s = seeds[i];
    const uint32_t km = seed_kmer(s), nb = g_tab_buckets[g];
    rep_flag_seed(seeds, i, s, km, tab + g_tab_off[g], nb, max_mult);
}

// the pairs of one block, selected in order (pair_owned_flag_kernel's flags, their scan), with their positions in the
// call's pair list
__global__ void pair_keep_pos_kernel(const unsigned long long *__restrict__ pairs, int64_t n_pairs,
                                     const uint32_t *__restrict__ flag, const uint32_t *__restrict__ pos,
                                     unsigned long long *__restrict__ out, uint32_t *__restrict__ out_pos) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs || !flag[t]) return;
    out[pos[t]] = pairs[t];
    out_pos[pos[t]] = (uint32_t)t;
}
// the position in the call's pair list of every edge of one block (edge_flag_kernel's flags, their scan): the key that
// merges the blocks' edges back into pair-list order
__global__ void edge_pos_kernel(const uint32_t *__restrict__ flag, const uint32_t *__restrict__ pos, int64_t n_pairs,
                                const uint32_t *__restrict__ pair_pos, uint32_t *__restrict__ edge_pos) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_pairs && flag[t]) edge_pos[pos[t]] = pair_pos[t];
}
__global__ void iota_u32_kernel(int64_t n, uint32_t *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = (uint32_t)t;
}
// out[t] = in[perm[t]] (edges and their --ci / --detailed records)
template <typename T>
__global__ void gather_kernel(const T *__restrict__ in, const uint32_t *__restrict__ perm, int64_t n, T *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = in[perm[t]];
}

}  // namespace skb
