// skani's -n on dist / search (skb_set_max_results, DESIGN.md section 3): keep each query's first N edges in the row
// order (query, ANI descending, reference ascending).  The edge list is sorted by (a << 32 | b), so two stable radix
// sorts -- on the ANI key, then on the query id -- give that order; an edge is kept when its rank in its query's run
// is below N, and the kept edges are compacted in their original (a, b) order.
#pragma once
#include "skb_common.cuh"

namespace skb {

// key: unsigned integers that sort like the ANI doubles, descending; idx: the edge's position
__global__ void best_n_key_kernel(const skb_edge *__restrict__ edges, int64_t n, unsigned long long *__restrict__ key,
                                  uint32_t *__restrict__ idx) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const unsigned long long u = (unsigned long long)__double_as_longlong(edges[t].ani);
    const unsigned long long asc = (u >> 63) ? ~u : (u | (1ull << 63));  // IEEE order -> unsigned order
    key[t] = ~asc;
    idx[t] = (uint32_t)t;
}

// the query id of the edge at every position of the ANI-sorted order
__global__ void best_n_query_kernel(const skb_edge *__restrict__ edges, const uint32_t *__restrict__ idx, int64_t n,
                                    uint32_t *__restrict__ query) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) query[t] = edges[idx[t]].b;
}

// query: the query ids in row order (runs of equal ids); position t has rank >= max_n in its run exactly when the
// position max_n before it holds the same query.  flag[] is indexed by the edge's original position.
__global__ void best_n_flag_kernel(const uint32_t *__restrict__ query, const uint32_t *__restrict__ idx, int64_t n,
                                   int64_t max_n, uint32_t *__restrict__ flag) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    flag[idx[t]] = (t < max_n || query[t - max_n] != query[t]) ? 1u : 0u;
}

// order-preserving compaction of one per-edge array under best_n_flag_kernel's flags and their exclusive scan
template <typename T>
__global__ void best_n_scatter_kernel(const T *__restrict__ in, int64_t n, const uint32_t *__restrict__ flag,
                                      const uint32_t *__restrict__ pos, T *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n && flag[t]) out[pos[t]] = in[t];
}

}  // namespace skb
