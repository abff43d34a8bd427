// skani's --full-matrix / --distance text (DESIGN.md section 3), rendered on the device one block of rows at a time:
// a dense cell -> edge map of the block (matrix_scatter_kernel), every row's byte length (matrix_row_len_kernel), an
// exclusive scan over the rows, then one CTA per row writes its label and cells at their offsets (matrix_write_kernel).
// A cell is the integer hundredths of its printed value (hundredths(), skb_common.cuh): 10000 on the diagonal, 0 for a
// pair that is not an edge, and for SKB_MATRIX_DISTANCE 10000 minus that.
#pragma once
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "skb_common.cuh"

namespace skb {

constexpr int MX_THREADS = 256;                   // one CTA per row
constexpr int MX_ITEMS = 4;                       // consecutive cells per thread and tile
constexpr int MX_TILE = MX_THREADS * MX_ITEMS;    // cells per tile
constexpr int MX_CELL_MAX = 16;                   // '\t', sign, the integer digits of any int32 / 100, '.', two digits

// cell (r, c) in hundredths; map_row: the cell -> edge index map of row r, -1 where no edge
__device__ __forceinline__ int matrix_cell(const int32_t *__restrict__ map_row, const skb_edge *__restrict__ edges,
                                           int32_t r, int32_t c, int32_t kind) {
    int v = 10000;
    if (c != r) {
        const int32_t e = map_row[c];
        v = 0;
        if (e >= 0) {
            const skb_edge &E = edges[e];
            v = (int)hundredths(kind == SKB_MATRIX_AF ? (E.a == (uint32_t)r ? E.af_a : E.af_b) : E.ani);
        }
    }
    return kind == SKB_MATRIX_DISTANCE ? 10000 - v : v;
}

// bytes of "\t%.2f" of v / 100
__device__ __forceinline__ uint32_t matrix_cell_width(int v) {
    uint32_t u = (uint32_t)(v < 0 ? -(int64_t)v : v) / 100, d = 1;
    while (u >= 10) {
        u /= 10;
        d++;
    }
    return 1 + (v < 0) + d + 3;
}

__device__ __forceinline__ void matrix_cell_text(char *p, int v, uint32_t w) {
    uint32_t u = (uint32_t)(v < 0 ? -(int64_t)v : v);
    p[0] = '\t';
    p[w - 1] = (char)('0' + u % 10);
    p[w - 2] = (char)('0' + u / 10 % 10);
    p[w - 3] = '.';
    u /= 100;
    int i = (int)w - 4;
    do {
        p[i--] = (char)('0' + u % 10);
        u /= 10;
    } while (u);
    if (v < 0) p[i] = '-';
}

// edge i fills cell (a - r0, b) when row a is in the block [r0, r0 + rows) and cell (b - r0, a) when row b is
__global__ void matrix_scatter_kernel(const skb_edge *__restrict__ edges, int64_t n_edges, int32_t n, int32_t r0,
                                      int32_t rows, int32_t *__restrict__ map) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_edges) return;
    const uint32_t a = edges[i].a, b = edges[i].b;
    if (a - (uint32_t)r0 < (uint32_t)rows) map[(size_t)(a - r0) * n + b] = (int32_t)i;
    if (b - (uint32_t)r0 < (uint32_t)rows) map[(size_t)(b - r0) * n + a] = (int32_t)i;
}

// row_len[k]: bytes of row r0 + k -- its label, its cells, the newline
__global__ void __launch_bounds__(MX_THREADS) matrix_row_len_kernel(const int32_t *__restrict__ map,
                                                                    const skb_edge *__restrict__ edges,
                                                                    const int64_t *__restrict__ label_off, int32_t n,
                                                                    int32_t r0, int32_t kind, uint64_t *__restrict__ row_len) {
    using Reduce = cub::BlockReduce<uint32_t, MX_THREADS>;
    __shared__ typename Reduce::TempStorage tmp;
    const int32_t r = r0 + (int32_t)blockIdx.x;
    const int32_t *row = map + (size_t)blockIdx.x * n;
    uint32_t w = 0;
    for (int32_t c = threadIdx.x; c < n; c += MX_THREADS) w += matrix_cell_width(matrix_cell(row, edges, r, c, kind));
    w = Reduce(tmp).Sum(w);
    if (threadIdx.x == 0) row_len[blockIdx.x] = (uint64_t)(label_off[r + 1] - label_off[r]) + w + 1;
}

// One CTA per row: the label, then tile by tile the cells -- widths block-scanned, text built in shared memory and
// stored in order -- then the newline, at row_off[k] of the block's text
__global__ void __launch_bounds__(MX_THREADS) matrix_write_kernel(const int32_t *__restrict__ map,
                                                                  const skb_edge *__restrict__ edges,
                                                                  const char *__restrict__ labels,
                                                                  const int64_t *__restrict__ label_off, int32_t n,
                                                                  int32_t r0, int32_t kind,
                                                                  const uint64_t *__restrict__ row_off,
                                                                  char *__restrict__ text) {
    using Scan = cub::BlockScan<uint32_t, MX_THREADS>;
    __shared__ typename Scan::TempStorage scan_tmp;
    __shared__ char tile[MX_TILE * MX_CELL_MAX];
    const int32_t r = r0 + (int32_t)blockIdx.x;
    const int32_t *row = map + (size_t)blockIdx.x * n;
    char *out = text + row_off[blockIdx.x];
    const int64_t l0 = label_off[r], ll = label_off[r + 1] - l0;
    for (int64_t i = threadIdx.x; i < ll; i += MX_THREADS) out[i] = labels[l0 + i];
    out += ll;
    for (int32_t t0 = 0; t0 < n; t0 += MX_TILE) {
        int v[MX_ITEMS];
        uint32_t w[MX_ITEMS], sum = 0;
#pragma unroll
        for (int j = 0; j < MX_ITEMS; j++) {
            const int32_t c = t0 + (int32_t)threadIdx.x * MX_ITEMS + j;
            v[j] = c < n ? matrix_cell(row, edges, r, c, kind) : 0;
            w[j] = c < n ? matrix_cell_width(v[j]) : 0;
            sum += w[j];
        }
        uint32_t off, total;
        Scan(scan_tmp).ExclusiveSum(sum, off, total);
#pragma unroll
        for (int j = 0; j < MX_ITEMS; j++) {
            if (w[j]) matrix_cell_text(tile + off, v[j], w[j]);
            off += w[j];
        }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < total; i += MX_THREADS) out[i] = tile[i];
        out += total;
        __syncthreads();  // the tile and the scan storage are reused
    }
    if (threadIdx.x == 0) *out = '\n';
}

}  // namespace skb
