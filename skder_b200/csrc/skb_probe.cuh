// K2 -- per-reference seed index: bucketed hash table keyed by the seed k-mer, and the batched anchor
// lookup the chunk kernel's P1 runs against it.
//
// Stand-in for skani's seed map (k-mer -> positions) used by the pairwise estimator behind
// `skani triangle|dist|search` (reference call sites src/skDER/skder.py:16-18, :58-59, :119).
//
// Layout: buckets of 4 slots = one 32-byte sector.  A k-mer has ONE home bucket; a record that finds it full
// raises the bucket's overflow flag and moves on to the next bucket, flagging every full bucket it passes.  A lookup
// reads the home bucket and goes on only while the bucket it has just read is flagged.  Tables are built at load
// factor 0.5 / 1 / 2 entries per bucket (the sparsest the device memory budget allows, skb_index): at 0.5 a present
// k-mer's bucket is flagged with probability 0.2%, so a lookup is ONE scattered sector read -- one L1 wavefront per
// lane instead of the two of the two-choice layout this replaces (ncu, round 1: l1tex data-pipe wavefronts 83% of
// peak, 2.3x the algorithmic bytes at L2) -- and the dependent second read is rare enough not to stall warps.
//
// Bit 1 of a table record (the repeat flag of the seed array, unused in the copies) carries two flags, both ACTIVE
// LOW so that an empty slot (all ones, the memset value) reads as "no flag":
//   slot 3     : 0 = the bucket overflowed (records continue in the next bucket);
//   slots 0..2 : 0 = this k-mer has more than one record in this genome (set by rep_flag_kernel in the k-mer's home
//                bucket).  A lookup that sees neither flag knows its home bucket holds at most one record of its
//                k-mer: the common path never counts hits (emit_anchors_narrow).
#pragma once
#include "skb_common.cuh"

namespace skb {

#ifndef SKB_PJ
#define SKB_PJ 4
#endif
constexpr int PJ = SKB_PJ;    // lookups in flight per lane in the batched probe
constexpr int STAGE_CAP = 8;  // hits staged per seed (max_mult upper bound)

__host__ __device__ inline uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }

__host__ __device__ inline uint32_t tab_home(uint32_t kmer, uint32_t nb) { return mulhi32(kmer * 0x9E3779B1u, nb); }
__host__ __device__ inline uint32_t tab_next(uint32_t b, uint32_t nb) { return b + 1 == nb ? 0 : b + 1; }
// slot 3 of a bucket flagged "records continue in the next bucket" (active low; an empty slot is all ones)
__host__ __device__ inline bool tab_flagged(uint64_t slot3) { return (slot3 & 2ull) == 0; }

__device__ __forceinline__ int genome_of(const uint64_t *__restrict__ off, int n, uint64_t i) {
    int lo = 0, hi = n - 1;  // last g with off[g] <= i
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// genome_of for a warp whose lanes hold consecutive, ascending i: lane 0 searches, the others walk on from there
// (a warp spans 32 records, a genome ~40,000).  All 32 lanes must call.
__device__ __forceinline__ int genome_of_warp(const uint64_t *__restrict__ off, int n, uint64_t i) {
    const uint64_t i0 = __shfl_sync(0xffffffffu, i, 0);
    int g = 0;
    if ((threadIdx.x & 31) == 0) g = genome_of(off, n, i0);
    g = __shfl_sync(0xffffffffu, g, 0);
    while (g + 1 < n && off[g + 1] <= i) g++;
    return g;
}

// insert one table record into the table T of nb buckets (64-bit CAS; no deletions ever)
__device__ __forceinline__ void tab_insert_rec(unsigned long long *T, uint32_t nb, unsigned long long rec) {
    uint32_t b = tab_home(seed_kmer(rec), nb);
    for (;;) {
        // occupancy from one 256-bit read (slots fill in order); .cg: other threads are inserting
        unsigned long long a[BUCKET];
        asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];"
                     : "=l"(a[0]), "=l"(a[1]), "=l"(a[2]), "=l"(a[3]) : "l"(T + (size_t)b * BUCKET) : "memory");
        int occ = 0;
#pragma unroll
        for (int k = 0; k < (int)BUCKET; k++) occ += a[k] != TAB_EMPTY;
        if (occ < (int)BUCKET) {
            if (atomicCAS(&T[(size_t)b * BUCKET + occ], (unsigned long long)TAB_EMPTY, rec) == TAB_EMPTY) return;
            continue;  // somebody else took the slot: look again
        }
        if (a[BUCKET - 1] & 2ull) atomicAnd(&T[(size_t)b * BUCKET + BUCKET - 1], ~2ull);
        b = tab_next(b, nb);
    }
}

// one thread per seed record: insert into its genome's table
__global__ void tab_insert_kernel(const uint64_t *__restrict__ seeds, uint64_t n_seeds,
                                  const uint64_t *__restrict__ g_seed_off, int n_genomes, uint64_t *tab,
                                  const uint64_t *__restrict__ g_tab_off, const uint32_t *__restrict__ g_tab_buckets,
                                  uint64_t first /* records [first, n_seeds) are inserted */) {
    uint64_t i = first + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int g = genome_of_warp(g_seed_off, n_genomes, i < n_seeds ? i : n_seeds - 1);
    if (i >= n_seeds) return;
    const uint32_t nb = g_tab_buckets[g];
    unsigned long long *T = reinterpret_cast<unsigned long long *>(tab + g_tab_off[g]);
    tab_insert_rec(T, nb, seeds[i] | 2ull);  // both table flags clear (active low)
}

struct Bucket {
    ulonglong2 lo, hi;  // slots 0..3
};
__device__ __forceinline__ Bucket empty_bucket() {
    Bucket B;
    B.lo = B.hi = make_ulonglong2(TAB_EMPTY, TAB_EMPTY);
    return B;
}
// One bucket = one 32-byte sector = ONE 256-bit load (LDG.E.256, sm_100).  Lookups are scattered, so every load
// instruction costs the L1 data pipe a wavefront per lane.  Buckets are 32-byte aligned (table offsets are
// multiples of BUCKET words, the allocation is 256-byte aligned).
__device__ __forceinline__ Bucket load_bucket(const uint64_t *__restrict__ T, uint32_t b) {
    Bucket B;
    const uint64_t *p = T + (size_t)b * BUCKET;
    asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(B.lo.x), "=l"(B.lo.y), "=l"(B.hi.x), "=l"(B.hi.y) : "l"(p));
    return B;
}

// entries holding `kmer` (an empty slot's k-mer field, all ones, is never a canonical k-mer)
__device__ __forceinline__ int tab_count(const uint64_t *__restrict__ T, uint32_t nb, uint32_t kmer, int cap) {
    uint32_t b = tab_home(kmer, nb);
    int c = 0;
    for (;;) {
        const Bucket B = load_bucket(T, b);
        c += (seed_kmer(B.lo.x) == kmer) + (seed_kmer(B.lo.y) == kmer) + (seed_kmer(B.hi.x) == kmer) + (seed_kmer(B.hi.y) == kmer);
        if (!tab_flagged(B.hi.y) || c >= cap) break;
        b = tab_next(b, nb);
    }
    return c;
}

// flag seed record i (s = seeds[i], km its k-mer) if its k-mer occurs more than max_mult times in its own genome (bit 1
// of the seed record), and mark the table records of every k-mer that occurs more than once (bit 1 of slots 0..2 of its
// home bucket, active low); T, nb: the genome's table
__device__ __forceinline__ void rep_flag_seed(uint64_t *seeds, uint64_t i, uint64_t s, uint32_t km, uint64_t *T, uint32_t nb,
                                              int max_mult) {
    const int c = tab_count(T, nb, km, max_mult + 1);
    if (c > max_mult) seeds[i] = s | 2ull;
    if (c > 1) {  // rare.  Only bit 1 changes, which no concurrent tab_count looks at
        unsigned long long *H = reinterpret_cast<unsigned long long *>(T) + (size_t)tab_home(km, nb) * BUCKET;
        for (int k = 0; k < (int)BUCKET - 1; k++) {
            const unsigned long long e = H[k];
            if (e != TAB_EMPTY && seed_kmer(e) == km && (e & 2ull)) atomicAnd(&H[k], ~2ull);
        }
    }
}

// rep_flag_seed for every seed record [first, n_seeds)
__global__ void rep_flag_kernel(uint64_t *seeds, uint64_t n_seeds, const uint64_t *__restrict__ g_seed_off,
                                int n_genomes, uint64_t *tab,
                                const uint64_t *__restrict__ g_tab_off, const uint32_t *__restrict__ g_tab_buckets,
                                int max_mult, uint64_t first) {
    uint64_t i = first + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int g = genome_of_warp(g_seed_off, n_genomes, i < n_seeds ? i : n_seeds - 1);
    if (i >= n_seeds) return;
    const uint64_t s = seeds[i];
    const uint32_t km = seed_kmer(s), nb = g_tab_buckets[g];
    uint64_t *T = tab + g_tab_off[g];
    rep_flag_seed(seeds, i, s, km, T, nb, max_mult);
}

// staged hit: (ref_pos << 1) | strand relation
__device__ __forceinline__ uint32_t enc_hit(uint64_t e, uint64_t sd) {
    return (seed_pos(e) << 1) | (uint32_t)(seed_strand(e) != seed_strand(sd));
}

// One lookup of the batch: lane's seed `sd` with its home bucket B already loaded.  Appends the
// seed's anchors (if it has 1..mult hits) after `base`; returns base + anchors of all 32 lanes.
__device__ __forceinline__ int probe_one(uint64_t sd, const Bucket &B, const uint64_t *__restrict__ T, uint32_t nb,
                                         int mult, int max_mult, int max_anchors, uint32_t *stage, uint64_t *anc,
                                         int base, int s, uint32_t cstart, int lane) {
    const uint32_t km = seed_kmer(sd);
    const uint64_t e4[4] = {B.lo.x, B.lo.y, B.hi.x, B.hi.y};
    // the k-mer is the top 30 bits of a record: compare on the high word only.  Flagged / out-of-range
    // lanes hold an all-empty bucket, whose k-mer field (all ones) is never a canonical k-mer.
    const uint32_t kmhi = km << 2;
    int c = 0;
    uint64_t e1 = 0;  // the hit when there is exactly one
#pragma unroll
    for (int x = 0; x < 4; x++) {
        const bool hit = (((uint32_t)(e4[x] >> 32)) ^ kmhi) < 4u;
        c += hit;
        if (hit) e1 = e4[x];
    }
    const bool spilled = tab_flagged(B.hi.y);  // rare: the k-mer's records may continue in the next bucket(s)
    const bool slow = spilled || c > 1;
    if (slow) {  // rare: repeats or spill -> stage all hits, sorted by ref position
        int cc = 0;
#pragma unroll
        for (int x = 0; x < 4; x++)
            if ((((uint32_t)(e4[x] >> 32)) ^ kmhi) < 4u) {
                if (cc < STAGE_CAP) stage[lane * STAGE_CAP + cc] = enc_hit(e4[x], sd);
                cc++;
            }
        if (spilled) {
            uint32_t b = tab_home(km, nb);
            for (;;) {
                b = tab_next(b, nb);
                const Bucket X = load_bucket(T, b);
                const uint64_t x4[4] = {X.lo.x, X.lo.y, X.hi.x, X.hi.y};
#pragma unroll
                for (int x = 0; x < 4; x++)
                    if (seed_kmer(x4[x]) == km) {
                        if (cc < STAGE_CAP) stage[lane * STAGE_CAP + cc] = enc_hit(x4[x], sd);
                        cc++;
                    }
                if (!tab_flagged(X.hi.y) || cc > max_mult) break;
            }
        }
        c = cc;
        if (c > mult) c = 0;
        for (int x = 1; x < c; x++) {  // insertion sort, c <= STAGE_CAP
            const uint32_t v = stage[lane * STAGE_CAP + x];
            int y = x - 1;
            while (y >= 0 && stage[lane * STAGE_CAP + y] > v) {
                stage[lane * STAGE_CAP + y + 1] = stage[lane * STAGE_CAP + y];
                y--;
            }
            stage[lane * STAGE_CAP + y + 1] = v;
        }
    }
    const uint64_t lowbits = ((uint64_t)(seed_pos(sd) - cstart) << 17) | (uint64_t)s;
    const unsigned any_slow = __ballot_sync(0xffffffffu, slow);
    if (!any_slow) {  // common: every lane has 0 or 1 hit -> offsets from one ballot
        const unsigned has = __ballot_sync(0xffffffffu, c == 1);
        if (c == 1) {
            const int dst = base + __popc(has & ((1u << lane) - 1u));
            const uint32_t v = enc_hit(e1, sd);
            if (dst < max_anchors) __stcg(anc + slab_off((uint32_t)dst), ((uint64_t)(v >> 1) << 32) | lowbits | ((uint64_t)(v & 1u) << 16));
        }
        return base + __popc(has);
    }
    int pre = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, pre, d);
        if (lane >= d) pre += u;
    }
    const int tot = __shfl_sync(0xffffffffu, pre, 31);
    pre -= c;
    if (!slow) {
        if (c == 1) {
            const uint32_t v = enc_hit(e1, sd);
            if (base + pre < max_anchors)
                __stcg(anc + slab_off((uint32_t)(base + pre)), ((uint64_t)(v >> 1) << 32) | lowbits | ((uint64_t)(v & 1u) << 16));
        }
    } else {
        for (int x = 0; x < c; x++) {
            const int dst = base + pre + x;
            const uint32_t v = stage[lane * STAGE_CAP + x];
            if (dst < max_anchors) __stcg(anc + slab_off((uint32_t)dst), ((uint64_t)(v >> 1) << 32) | lowbits | ((uint64_t)(v & 1u) << 16));
        }
    }
    return base + tot;
}

// first batch of a task's seed records (PJ x 32), one per lane and slot; out-of-range = flagged record
__device__ __forceinline__ void load_first_batch(const uint64_t *__restrict__ qs, int nseeds, int lane, uint64_t (&sdn)[PJ]) {
#pragma unroll
    for (int j = 0; j < PJ; j++) {
        const int s = 32 * j + lane;
        sdn[j] = s < nseeds ? qs[s] : 2ull;  // rep bit set = skip
    }
}

// sdn holds this task's first batch on entry and the NEXT task's first batch (qs_next/ns_next) on exit,
// so the only latency a task exposes is that of its bucket reads.
__device__ __forceinline__ int emit_anchors(const uint64_t *__restrict__ qs, int nseeds, uint32_t cstart,
                                            const uint64_t *__restrict__ T, uint32_t nb, int mult, int max_mult,
                                            int max_anchors, uint32_t *stage, uint64_t *anc, int lane,
                                            uint64_t (&sdn)[PJ], const uint64_t *__restrict__ qs_next, int ns_next) {
    int base = 0;
    for (int s0 = 0; s0 < nseeds; s0 += 32 * PJ) {
        uint64_t sd[PJ];
        Bucket B[PJ];
#pragma unroll
        for (int j = 0; j < PJ; j++) {
            sd[j] = sdn[j];
            B[j] = seed_rep(sd[j]) ? empty_bucket() : load_bucket(T, tab_home(seed_kmer(sd[j]), nb));
        }
        if (s0 + 32 * PJ < nseeds) {
#pragma unroll
            for (int j = 0; j < PJ; j++) {
                const int s = s0 + 32 * PJ + 32 * j + lane;
                sdn[j] = s < nseeds ? qs[s] : 2ull;
            }
        } else
            load_first_batch(qs_next, ns_next, lane, sdn);
#pragma unroll
        for (int j = 0; j < PJ; j++) {
            if (s0 + 32 * j >= nseeds) break;  // warp-uniform
            base = probe_one(sd[j], B[j], T, nb, mult, max_mult, max_anchors, stage, anc, base, s0 + 32 * j + lane,
                             cstart, lane);
        }
    }
    return base;
}

// ---- NARROW variant: every padded position of the database is below 2^30 - 2^21 (skb_api.cu picks it per call; any
// bacterial set qualifies).  Then the high word of a seed record is exactly kmer << 2 and the low word holds the whole
// position, so a slot matches iff its high word EQUALS the query seed's, positions and strands come from the low words
// alone, and -- thanks to the two table flags -- the common path never counts hits: no flag seen means the home bucket
// holds at most one record of the k-mer.  ~45 instructions per 32 lookups instead of ~115 (ncu source page, round 2:
// the kernel issues 67 % of peak and is bound by instruction count, not by L2 or DRAM).
__device__ __forceinline__ Bucket load_bucket_if(const uint64_t *__restrict__ T, uint32_t b, bool valid) {
    Bucket B;  // left undefined for lanes that do not look up: every use below is guarded by `valid`
    const uint64_t *p = T + (size_t)b * BUCKET;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %5, 0;\n\t@p ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];\n\t}"
                 : "=l"(B.lo.x), "=l"(B.lo.y), "=l"(B.hi.x), "=l"(B.hi.y) : "l"(p), "r"((int)valid));
    return B;
}

__device__ __forceinline__ int probe_narrow(uint2 sd, Bucket &B, const uint64_t *__restrict__ T,
                                            uint32_t nb, int mult, int max_mult, int max_anchors, uint32_t *stage,
                                            uint64_t *anc, int base, int s, uint32_t cstart, int lane) {
    const bool valid = !(sd.x & 2u);  // not a repeat, not past the chunk's end: B was loaded
    const uint32_t l3 = (uint32_t)B.hi.y;
    const bool h0 = valid && (uint32_t)(B.lo.x >> 32) == sd.y, h1 = valid && (uint32_t)(B.lo.y >> 32) == sd.y;
    const bool h2 = valid && (uint32_t)(B.hi.x >> 32) == sd.y, h3 = valid && (uint32_t)(B.hi.y >> 32) == sd.y;
    const bool any = h0 || h1 || h2 || h3;
    // first hit in slot order; slot 3's bit 1 is the overflow flag, not a repeat flag
    uint32_t e = l3 | 2u;  // predicated moves, not a branch per slot
    if (h2) e = (uint32_t)B.hi.x;
    if (h1) e = (uint32_t)B.lo.y;
    if (h0) e = (uint32_t)B.lo.x;
    const bool slow = (any && !(e & 2u)) || (valid && !(l3 & 2u));
    if (__any_sync(0xffffffffu, slow)) {  // repeats or an overflowed bucket somewhere in the warp: the general code
        if (!valid) B = empty_bucket();  // in place: the caller is done with this bucket
        return probe_one(((uint64_t)sd.y << 32) | sd.x, B, T, nb, mult, max_mult, max_anchors, stage, anc, base, s, cstart, lane);
    }
    const unsigned has = __ballot_sync(0xffffffffu, any);
    if (any) {
        const int dst = base + __popc(has & ((1u << lane) - 1u));
        if (dst < max_anchors) {
            const uint32_t lo = (((sd.x >> 2) - cstart) << 17) | (((e ^ sd.x) & 1u) << 16) | (uint32_t)s;
            __stcg(anc + slab_off((uint32_t)dst), ((uint64_t)(e >> 2) << 32) | (uint64_t)lo);
        }
    }
    return base + __popc(has);
}

__device__ __forceinline__ void load_first_batch_narrow(const uint2 *__restrict__ qs, int nseeds, int lane, uint2 (&sdn)[PJ]) {
#pragma unroll
    for (int j = 0; j < PJ; j++) {
        const int s = 32 * j + lane;
        sdn[j] = s < nseeds ? qs[s] : make_uint2(2u, 0u);  // rep bit set = skip
    }
}

// same contract as emit_anchors
__device__ __forceinline__ int emit_anchors_narrow(const uint2 *__restrict__ qs, int nseeds, uint32_t cstart,
                                                   const uint64_t *__restrict__ T, uint32_t nb, int mult, int max_mult,
                                                   int max_anchors, uint32_t *stage, uint64_t *anc, int lane,
                                                   uint2 (&sdn)[PJ], const uint2 *__restrict__ qs_next, int ns_next) {
    int base = 0;
    for (int s0 = 0; s0 < nseeds; s0 += 32 * PJ) {
        uint2 sd[PJ];
        Bucket B[PJ];
#pragma unroll
        for (int j = 0; j < PJ; j++) {
            sd[j] = sdn[j];
            B[j] = load_bucket_if(T, tab_home(sd[j].y >> 2, nb), !(sd[j].x & 2u));
        }
        if (s0 + 32 * PJ < nseeds) {
            const uint2 *qn = qs + s0 + 32 * PJ + lane;
#pragma unroll
            for (int j = 0; j < PJ; j++) sdn[j] = s0 + 32 * PJ + 32 * j + lane < nseeds ? qn[32 * j] : make_uint2(2u, 0u);
        } else
            load_first_batch_narrow(qs_next, ns_next, lane, sdn);
#pragma unroll
        for (int j = 0; j < PJ; j++) {
            if (s0 + 32 * j >= nseeds) break;  // warp-uniform
            base = probe_narrow(sd[j], B[j], T, nb, mult, max_mult, max_anchors, stage, anc, base, s0 + 32 * j + lane,
                                cstart, lane);
        }
    }
    return base;
}

}  // namespace skb
