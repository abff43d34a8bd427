// K1 -- FracMinHash sketching kernel (seeds k=15 c=125, markers k=21 c=m: 1000 unless skb_set_marker_compression).
//
// Stands in for skani's sketching pass, reached from skDER at src/skDER/skder.py:16 (triangle),
// :58 (dist), :103 (sketch) and :119 (search).  Bit-exact against oracle/skani_oracle.c
// sketch_contig().
//
// Layout: a genome is its kept contigs concatenated, 2 bits/base, 32 bases per 64-bit word, base j
// in bits 2*(j%32).  One lane owns 64 consecutive bases = ONE 128-bit load, a warp 2048 bases
// (512 contiguous bytes per request), a CTA 16384.  The 20 bases of left context come from the
// neighbouring lane by shuffle (lane 0 re-reads one word).  Phase A rolls the forward and
// reverse-complement 21-mer windows and hashes both k-mers at every valid position, keeping two
// 64-bit hit masks; the hash pass stores them (16 bytes per lane) next to the per-warp counts, and
// the emit pass -- after the counts are scanned -- reads the masks back instead of hashing again and
// turns the mask bits into records at offsets fixed by a warp prefix sum + the scanned per-warp
// counts, so seeds come out in position order with no sort.
#pragma once
#include "skb_common.cuh"

namespace skb {

constexpr int SK_WARPS = 8;
constexpr int SK_THREADS = SK_WARPS * 32;
constexpr int SK_LANE_BASES = 64;
constexpr int SK_WARP_BASES = 32 * SK_LANE_BASES;         // 2048
constexpr int SK_TILE_BASES = SK_WARPS * SK_WARP_BASES;   // 16384

struct SketchBatch {
    const uint64_t *packed;      // all genomes of the batch, each starting on an even word
    const uint64_t *g_word_off;  // [n+1]
    const uint64_t *g_nbases;    // [n]
    const uint32_t *g_ctg_off;   // [n+1] into ctg_start; per-sequence mode: also the batch-local id of each file's first record
    const uint64_t *ctg_start;   // unpadded first-base offset of each contig inside its genome
    const uint32_t *tile_off;    // [n+1] CTA-tile prefix sum
    int32_t n;
    uint32_t first_gid;          // DB id of batch genome 0
    uint64_t thr_marker;         // a canonical 21-mer is a marker iff its hash is below this (marker_threshold)
};

// reverse the order of the 21 two-bit groups held in the low 42 bits of x
__device__ __forceinline__ uint64_t rev2_42(uint64_t x) {
    uint64_t y = __brevll(x);  // bit-reverse: group order reversed, bits inside each group swapped
    y = ((y >> 1) & 0x5555555555555555ull) | ((y & 0x5555555555555555ull) << 1);
    return y >> (64 - 2 * K_MARKER);
}

// reverse the order of the 16 two-bit groups of a 32-bit word
__device__ __forceinline__ uint32_t rev2_32(uint32_t x) {
    const uint32_t y = __brev(x);
    return ((y >> 1) & 0x55555555u) | ((y & 0x55555555u) << 1);
}

// PER_SEQ (emit pass only; skb_add_sequences): every contig of a batch entry is its own genome -- its marker keys carry
// the genome id first_gid + g_ctg_off[g] + ci and its seeds the record-local position p - ctg_start[ci] (contig index
// 0), which is what the same record sketched as a one-contig genome gets.  The hash pass does not depend on the mode.
template <bool EMIT, bool PER_SEQ = false>
__global__ void __launch_bounds__(SK_THREADS)
sketch_kernel(SketchBatch b, uint32_t *__restrict__ warp_seed_cnt, uint32_t *__restrict__ warp_marker_cnt,
              const uint32_t *__restrict__ warp_seed_off, const uint32_t *__restrict__ warp_marker_off,
              uint64_t *__restrict__ seeds_out, uint64_t *__restrict__ mkeys_out, ulonglong2 *__restrict__ masks) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // genome of this CTA: last g with tile_off[g] <= blockIdx.x
    int lo = 0, hi = b.n - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (b.tile_off[mid] <= blockIdx.x)
            lo = mid;
        else
            hi = mid - 1;
    }
    const int g = lo;
    const uint64_t nb = b.g_nbases[g];
    const uint64_t *W = b.packed + b.g_word_off[g];
    const uint64_t nwords = b.g_word_off[g + 1] - b.g_word_off[g];
    const uint64_t tile = blockIdx.x - b.tile_off[g];
    const uint64_t p0 = tile * SK_TILE_BASES + (uint64_t)warp * SK_WARP_BASES + (uint64_t)lane * SK_LANE_BASES;
    const size_t wgid = (size_t)blockIdx.x * SK_WARPS + warp;

    const uint64_t widx = p0 >> 5;
    ulonglong2 v = make_ulonglong2(0ull, 0ull);
    if (widx < nwords) v = *reinterpret_cast<const ulonglong2 *>(W + widx);  // nwords is even
    uint64_t prevw = __shfl_up_sync(0xffffffffu, v.y, 1);
    if (lane == 0) prevw = (widx > 0 && widx <= nwords) ? W[widx - 1] : 0ull;

    uint64_t seed_mask = 0, marker_mask = 0;
    // contig bookkeeping
    const uint64_t *cs = b.ctg_start + b.g_ctg_off[g];
    const int nc = (int)(b.g_ctg_off[g + 1] - b.g_ctg_off[g]);
    int ci0 = 0;
    if (EMIT) {  // the hash pass left this lane's two hit masks behind: no second round of hashing
        const ulonglong2 mk = masks[wgid * 32 + lane];
        seed_mask = mk.x;
        marker_mask = mk.y;
    }
    if (p0 < nb && (!EMIT || (seed_mask | marker_mask) != 0)) {
        int l2 = 0, h2 = nc - 1;  // last contig with start <= p0
        while (l2 < h2) {
            int mid = (l2 + h2 + 1) >> 1;
            if (cs[mid] <= p0)
                l2 = mid;
            else
                h2 = mid - 1;
        }
        ci0 = l2;
    }
    if (!EMIT && p0 < nb) {
        // The 21-mer ending at lane-local base j is a 42-bit window of the lane's 192-bit string (prevw, v.x, v.y)
        // at bit 24 + 2j: complemented it IS the rolling reverse-complement value; the rolling forward value is the
        // same window with its base order reversed, i.e. a window of the base-reversed string at bit 126 - 2j.
        // So nothing rolls: per position two funnel-shift extractions with compile-time shifts (16 positions
        // unrolled, the 32-bit words rotate between blocks), 32-bit arithmetic for the 30-bit seed, and no
        // per-position contig bookkeeping -- every position is hashed and the invalid ones (past the genome end,
        // or within 20 bases after a contig start) are cleared from the masks afterwards.
        uint32_t a0 = (uint32_t)prevw, a1 = (uint32_t)(prevw >> 32), a2 = (uint32_t)v.x, a3 = (uint32_t)(v.x >> 32),
                 a4 = (uint32_t)v.y, a5 = (uint32_t)(v.y >> 32);
        uint32_t b0 = rev2_32(a5), b1 = rev2_32(a4), b2 = rev2_32(a3), b3 = rev2_32(a2), b4 = rev2_32(a1), b5 = rev2_32(a0);
#pragma unroll 1
        for (int jb = 0; jb < SK_LANE_BASES / 16; jb++) {
            uint32_t sm16 = 0, mm16 = 0;
#pragma unroll
            for (int u = 0; u < 16; u++) {
                // reverse-complement window: ~(a >> (24 + 2u)), 42 bits
                constexpr int HI10 = (1 << (2 * K_MARKER - 32)) - 1;
                const int sh = 24 + 2 * u;
                uint32_t xlo, xhi;
                if (sh < 32) {
                    xlo = __funnelshift_r(a0, a1, sh);
                    xhi = __funnelshift_r(a1, a2, sh);
                } else {
                    xlo = __funnelshift_r(a1, a2, sh - 32);
                    xhi = a2 >> (sh - 32);
                }
                const uint32_t rlo = ~xlo, rhi = ~xhi & HI10;
                // forward window: b >> (30 - 2u) with b0..b2 = words 3-jb .. 5-jb of the reversed string
                const int sf = 30 - 2 * u;
                const uint32_t flo = __funnelshift_r(b3, b4, sf);
                const uint32_t fhi = __funnelshift_r(b4, b5, sf) & HI10;
                // seed: last 15 bases = low 30 bits of f, top 30 bits of r
                const uint32_t fs = flo & (uint32_t)MASK_SEED;
                const uint32_t rs = __funnelshift_r(rlo, rhi, 2 * (K_MARKER - K_SEED));
                const uint32_t cseed = fs < rs ? fs : rs;
                if (mm_hash64((uint64_t)cseed) < THR_SEED) sm16 |= 1u << u;
                const uint64_t f = ((uint64_t)fhi << 32) | flo, r = ((uint64_t)rhi << 32) | rlo;
                const uint64_t cm = f < r ? f : r;
                if (mm_hash64(cm) < b.thr_marker) mm16 |= 1u << u;
            }
            seed_mask |= (uint64_t)sm16 << (16 * jb);
            marker_mask |= (uint64_t)mm16 << (16 * jb);
            a0 = a1, a1 = a2, a2 = a3, a3 = a4, a4 = a5, a5 = 0;
            b5 = b4, b4 = b3, b3 = b2, b2 = b1, b1 = b0, b0 = 0;
        }
        // valid positions: inside the genome, and a full 21-mer inside one contig
        const uint64_t left = nb - p0;
        uint64_t valid = left >= 64 ? ~0ull : ((1ull << left) - 1);
        for (int k = ci0; k < nc; k++) {
            const int64_t lo = (int64_t)cs[k] - (int64_t)p0;  // contig start relative to the lane
            if (lo >= SK_LANE_BASES) break;
            const int64_t hi = lo + (K_MARKER - 1);
            if (hi <= 0) continue;
            const int l = lo < 0 ? 0 : (int)lo, h = hi > SK_LANE_BASES ? SK_LANE_BASES : (int)hi;
            const uint64_t span = (h - l) >= 64 ? ~0ull : ((1ull << (h - l)) - 1);
            valid &= ~(span << l);
        }
        seed_mask &= valid;
        marker_mask &= valid;
    }
    const int ns = __popcll(seed_mask), nm = __popcll(marker_mask);
    if (!EMIT) {
        masks[wgid * 32 + lane] = make_ulonglong2(seed_mask, marker_mask);
        const unsigned ts = __reduce_add_sync(0xffffffffu, (unsigned)ns);
        const unsigned tm = __reduce_add_sync(0xffffffffu, (unsigned)nm);
        if (lane == 0) {
            warp_seed_cnt[wgid] = ts;
            warp_marker_cnt[wgid] = tm;
        }
        return;
    } else {
        // exclusive prefix over lanes
        int ps = ns, pm = nm;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int ts = __shfl_up_sync(0xffffffffu, ps, d), tm = __shfl_up_sync(0xffffffffu, pm, d);
            if (lane >= d) {
                ps += ts;
                pm += tm;
            }
        }
        size_t so = (size_t)warp_seed_off[wgid] + (ps - ns);
        size_t mo = (size_t)warp_marker_off[wgid] + (pm - nm);
        if ((seed_mask | marker_mask) == 0) return;
        const uint64_t gid = PER_SEQ ? (uint64_t)b.first_gid + b.g_ctg_off[g] : (uint64_t)b.first_gid + g;
        int ci = ci0;
        uint64_t hits = seed_mask | marker_mask;
        while (hits) {
            const int j = __ffsll((long long)hits) - 1;
            hits &= hits - 1;
            const uint64_t p = p0 + j;
            while (ci + 1 < nc && cs[ci + 1] <= p) ci++;
            // 21-mer ending at lane-local base j from the 192-bit string (prevw, v.x, v.y): starts at bit 24+2j
            const int s = 64 + 2 * j - 2 * (K_MARKER - 1);
            const int wi = s >> 6, sh = s & 63;
            const uint64_t w0 = wi == 0 ? prevw : (wi == 1 ? v.x : v.y);
            const uint64_t w1 = wi == 0 ? v.x : v.y;  // wi == 2 never needs w1 (sh + 42 <= 64 there)
            uint64_t x = w0 >> sh;
            if (sh > 64 - 2 * K_MARKER) x |= w1 << (64 - sh);
            x &= MASK_MARKER;                 // base (j-20) in bits 0-1 ... base j in bits 40-41
            const uint64_t r = (~x) & MASK_MARKER;  // == rolling reverse-complement window
            const uint64_t f = rev2_42(x);          // == rolling forward window
            if ((seed_mask >> j) & 1) {
                const uint64_t fs = f & MASK_SEED, rs = r >> (2 * (K_MARKER - K_SEED));
                const int fwd = fs < rs;
                const uint64_t cseed = fwd ? fs : rs;
                const uint64_t ppos = PER_SEQ ? p - cs[ci] : p + (uint64_t)ci * CONTIG_PAD;
                seeds_out[so++] = (cseed << 34) | (ppos << 2) | (uint64_t)fwd;
            }
            if ((marker_mask >> j) & 1) {
                const uint64_t cm = f < r ? f : r;
                mkeys_out[mo++] = (cm << GID_BITS) | (PER_SEQ ? gid + ci : gid);
            }
        }
    }
}

// out[i] = src[idx[i] * mult]: the scanned per-warp offsets at every genome's first tile
__global__ void gather_strided_kernel(const uint32_t *__restrict__ src, const uint32_t *__restrict__ idx, uint32_t mult,
                                      int n, uint32_t *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[(size_t)idx[i] * mult];
}

// Per-sequence mode: out[r] = batch-local offset of the first seed of contig r of the batch (ctg_start order), and
// out[n_rec] = the batch's seed total.  Seeds come out in position order, so a contig's seeds start where the seeds
// before its first base end: the scanned offset of the warp holding that base plus the seed bits the hash pass left in
// the masks of the lanes, and the bits of its own lane, before it.
__global__ void record_seed_off_kernel(SketchBatch b, const uint32_t *__restrict__ warp_seed_off,
                                       const ulonglong2 *__restrict__ masks, int n_rec, size_t n_warps,
                                       uint32_t *__restrict__ out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r == 0) out[n_rec] = warp_seed_off[n_warps];
    if (r >= n_rec) return;
    int lo = 0, hi = b.n - 1;  // batch entry of contig r: last g with g_ctg_off[g] <= r
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (b.g_ctg_off[mid] <= (uint32_t)r)
            lo = mid;
        else
            hi = mid - 1;
    }
    const uint64_t s = b.ctg_start[r];
    const size_t wgid = ((size_t)b.tile_off[lo] + s / SK_TILE_BASES) * SK_WARPS + (s % SK_TILE_BASES) / SK_WARP_BASES;
    const int lane = (int)((s % SK_WARP_BASES) / SK_LANE_BASES), j = (int)(s % SK_LANE_BASES);
    uint32_t o = warp_seed_off[wgid];
    for (int l = 0; l < lane; l++) o += __popcll(masks[wgid * 32 + l].x);
    out[r] = o + __popcll(masks[wgid * 32 + lane].x & ((1ull << j) - 1));
}

}  // namespace skb
