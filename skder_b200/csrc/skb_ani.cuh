// K4 -- seed anchoring + per-chunk chaining (chunk kernel), chain selection + ANI/AF (finalize kernel).
//
// Stands in for skani's pairwise estimator behind `skani triangle|dist|search`
// (reference call sites src/skDER/skder.py:16-18, :58-59, :119).  Integer results (anchors, seeds,
// spans, chain count) are bit-exact against oracle/skani_oracle.c ora_pair(); ANI/AF are the same
// IEEE double expressions (device pow() may differ from glibc's in the last ulp).
//
// A task = (surviving pair, 20 kb query chunk).  Kernels, each at the occupancy its bottleneck wants; anchors and
// DP results go through a scratch array in HBM (written once, read once: the 2*16*A term of the roofline model).
//   K4a anchor_kernel (warp per task, 3 CTAs of 8 warps per SM, tasks grabbed 8 at a time): streams the chunk's
//      position-ordered seeds (coalesced 8-byte records), probes the reference's bucketed hash index (L2-resident: a
//      clade's members all hit the same tables) and writes the anchors in QUERY order -- the order the DP wants, so
//      there is no sort.  Bound by the L1 data pipe: every lookup is one scattered 32-byte sector.
//   K4b chain_kernel (thread per task): the chaining DP.  The two nearest predecessors live in registers, the rest
//      of the 16-anchor look-back window in a shared-memory ring that only the two uncommon paths read -- and those
//      are served by the whole warp (lane d takes window entry d).  It also tracks the best end of every DP tree and
//      writes the chunk's top candidates itself.
//   K4c ends_kernel (warp per task): the chunks with more DP trees than chain_kernel tracks (a compact list): best
//      end of every tree with >= min_anchors / min_score; the chunk's top `max_chunk_chains` by (score, q0, r0).
//   cand_pack_kernel + finalize_warp_kernel: chains packed into per-pair lists (extension precomputed); ONE WARP per
//      pair orders them, finds the chains that touch, resolves the greedy non-overlap selection over those only, sums
//      anchors, seeds and the symmetrically clipped spans of the accepted chains, and writes
//      ANI = ((A - 2n) / (S - 2n))^(1/15) (n chains, end anchors left out), AF = span / genome length.
//   finalize_kernel: one CTA per pair, for the pairs the warp kernel lists (more candidates than its shared memory
//      takes, or many blocking relations); beyond MAXP candidates the same code runs on global scratch
//      (finalize_kernel<true>).  No pair is capped or dropped.
#pragma once
#include <type_traits>

#include "skb_common.cuh"
#include "skb_index.cuh"

namespace skb {

constexpr int LB = 16;                        // DP look-back in anchors
constexpr int DP_UNR = 4;                     // anchors fetched per DP iteration (one 32-byte sector)
#ifndef SKB_DP_BODY
#define SKB_DP_BODY 2
#endif
constexpr int DP_BODY = SKB_DP_BODY;          // copies of the DP step in the loop body (2 or 4): code size vs loop overhead
constexpr int DIAG_SLACK = 64;                // chain_kernel short cut: diagonal drift followed without a rebuild
constexpr int NEG_F = -(1 << 24);             // DP score of an empty window slot
constexpr int ANC_THREADS = 256;              // K4a: 8 warps = 8 tasks per CTA pass
constexpr int DP_THREADS = 128;               // K4b: one task per thread
constexpr int END_THREADS = 256;              // K4c: 8 warps = 8 tasks per CTA pass
constexpr int MAXA = SLAB;                    // anchors per chunk (256)
constexpr int MAXP = 4096;                    // chain candidates per pair the shared-memory finalize kernel takes
constexpr int STAGE = 8;                      // max_mult upper bound (hits staged per seed)
constexpr int ENDS_K = 8;                     // qualifying DP trees per chunk tracked inside chain_kernel
constexpr int SLOTS = 8;                      // candidate slots per task (max_chunk_chains upper bound)
constexpr int FIN_THREADS = 256;

struct AniParams {
    int32_t band_bp, max_gap, anchor_score, min_anchors, min_score, max_mult, max_chunk_chains;
    int32_t ovl_num, ovl_den, span_ext;
    double debias_a, debias_g;
};

struct PairInfo {
    uint32_t q, r;  // query / reference genome ids
    uint32_t swapped;
    uint32_t nch;   // chunks of the query
};

// anchor record: ref_pos(32) | q_rel(15) | rev(1) | seed index in chunk(16)
__device__ __forceinline__ uint32_t an_r(uint64_t a) { return (uint32_t)(a >> 32); }
__device__ __forceinline__ uint32_t an_q(uint64_t a) { return ((uint32_t)a >> 17) & 0x7fffu; }
__device__ __forceinline__ uint32_t an_rev(uint64_t a) { return ((uint32_t)a >> 16) & 1u; }
__device__ __forceinline__ uint32_t an_sidx(uint64_t a) { return (uint32_t)a & 0xffffu; }
// DP result record: f(13) << 17 | root(8) << 9 | cnt(9)
__device__ __forceinline__ uint32_t rs_f(uint32_t x) { return x >> 17; }
__device__ __forceinline__ uint32_t rs_root(uint32_t x) { return (x >> 9) & 0xffu; }
__device__ __forceinline__ uint32_t rs_cnt(uint32_t x) { return x & 0x1ffu; }

struct __align__(16) Cand {
    uint32_t q0, q1, r0, r1;
    uint32_t chunk;
    uint16_t score, n_anchors;
    uint16_t n_seeds;
    uint8_t ordinal, rev;
    uint32_t pad;
};
static_assert(sizeof(Cand) == 32, "cand size");
static_assert(STAGE == STAGE_CAP, "stage layout");

// roles + sort key per pair (one thread per pair)
__global__ void pair_setup_kernel(DbView db, const unsigned long long *__restrict__ pairs, int64_t n_pairs,
                                  PairInfo *__restrict__ info, unsigned long long *__restrict__ sort_key,
                                  uint32_t *__restrict__ idx) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const uint32_t ga = (uint32_t)(pairs[p] >> 32), gb = (uint32_t)(pairs[p] & 0xffffffffu);
    const uint64_t nsa = db.g_seed_off[ga + 1] - db.g_seed_off[ga];
    const uint64_t nsb = db.g_seed_off[gb + 1] - db.g_seed_off[gb];
    PairInfo pi;
    pi.swapped = nsb < nsa;  // query = genome with fewer seeds (ties: a)
    pi.q = pi.swapped ? gb : ga;
    pi.r = pi.swapped ? ga : gb;
    pi.nch = db.g_chunk_off[pi.q + 1] - db.g_chunk_off[pi.q];
    info[p] = pi;
    sort_key[p] = ((unsigned long long)pi.r << 32) | pi.q;  // pairs sharing a reference index run together (L2 reuse)
    idx[p] = (uint32_t)p;
}

// pairs in reference-major order: info_sorted[i] = info[perm[i]]
__global__ void pair_gather_kernel(const PairInfo *__restrict__ info, const uint32_t *__restrict__ perm, int64_t n_pairs,
                                   PairInfo *__restrict__ info_sorted, uint32_t *__restrict__ nch_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const PairInfo pi = info[perm[i]];
    info_sorted[i] = pi;
    nch_out[i] = pi.nch;
}

// task descriptors: the (pair, chunk) decode is a chain of ~20 dependent loads, so it is done once,
// one thread per task, instead of by every warp in front of its two useful loads
struct __align__(16) TaskDesc {
    uint64_t seed_idx;  // first seed record of the chunk (index into db.seeds)
    uint64_t tab_idx;   // first slot of the reference's table (index into db.tab)
    uint32_t nseeds, cstart, nb, ch;
};
static_assert(sizeof(TaskDesc) == 32, "desc size");

// task_off: GLOBAL exclusive scan of the chunk counts, pointing at this batch's first pair; base = its value there
__global__ void task_setup_kernel(DbView db, const PairInfo *__restrict__ info, const uint32_t *__restrict__ task_off,
                                  uint32_t base, int64_t n_pairs, uint32_t n_tasks, TaskDesc *__restrict__ desc,
                                  uint32_t *__restrict__ task_pair) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tasks) return;
    int64_t lo = 0, hi = n_pairs - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (task_off[mid] - base <= t)
            lo = mid;
        else
            hi = mid - 1;
    }
    const PairInfo pi = info[lo];
    TaskDesc d;
    d.ch = t - (task_off[lo] - base);
    const uint32_t choff = db.g_chunk_off[pi.q];
    const uint32_t *cbeg = db.chunk_begin + choff + pi.q;
    const uint32_t sb = cbeg[d.ch];
    d.nseeds = cbeg[d.ch + 1] - sb;
    d.seed_idx = db.g_seed_off[pi.q] + sb;
    d.cstart = db.chunk_start[choff + d.ch];
    d.tab_idx = db.g_tab_off[pi.r];
    d.nb = db.g_tab_buckets[pi.r];
    desc[t] = d;
    task_pair[t] = (uint32_t)lo;
}

// ---- K4a: anchors.  One warp per task; the only dependent reads are descriptor -> seed records ->
// buckets, covered by the other resident warps.
// 3 CTAs of 8 warps per SM = 80 registers per thread: at 4 (64 registers) the four buckets in flight per lane spill,
// and local-memory traffic competes for the very L1 data pipe the scattered bucket reads are bound by (round 2 A/B on
// config3: 5.0 ms per launch at 3 CTAs without spills, 6.8 ms at 4 CTAs with 124 bytes of spill stores).
#ifndef SKB_ANC_MIN_CTAS
#define SKB_ANC_MIN_CTAS 3
#endif
#ifndef SKB_ANC_GRAB
#define SKB_ANC_GRAB 8
#endif
constexpr int ANC_GRAB = SKB_ANC_GRAB;  // consecutive tasks a warp takes from the counter at a time (<= 32)

template <bool NARROW>
__global__ void __launch_bounds__(ANC_THREADS, SKB_ANC_MIN_CTAS)
anchor_kernel(DbView db, AniParams prm, const TaskDesc *__restrict__ desc, uint32_t n_tasks,
              uint64_t *__restrict__ anc_all, uint16_t *__restrict__ task_n, uint32_t *__restrict__ next_task) {
    __shared__ uint32_t stage_all[ANC_THREADS / 32][32 * STAGE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *stage = stage_all[warp];
    __shared__ TaskDesc sdesc_all[ANC_THREADS / 32][ANC_GRAB];
    TaskDesc *sdesc = sdesc_all[warp];
    using seed_t = typename std::conditional<NARROW, uint2, uint64_t>::type;
    // Tasks are handed out in order from one counter, not strided by CTA: the grid is persistent and, next to the
    // consumer kernels of the previous batch, its CTAs become resident at different times; a CTA that starts late
    // must join the others on the reference tables that are in L2 NOW (tasks are reference-major), not work
    // through a fixed share milliseconds behind them (measured: 11 ms -> 54 ms per launch with a strided loop).
    // A warp takes ANC_GRAB consecutive tasks per visit to the counter: counter -> descriptor -> seed records ->
    // buckets is a chain of four dependent round trips of ~1 us each against ~0.4 us of instructions per task (ncu,
    // round 2: 41 % of the stall samples on the long scoreboard at 67 % issue).  With a grab the first two are paid
    // once per ANC_GRAB tasks (the descriptors wait in shared memory), and the first seed records of the next task
    // are fetched while the current task's last buckets are in flight (emit_anchors' qs_next).
    for (;;) {
        uint32_t t0 = 0;
        if (lane == 0) t0 = atomicAdd(next_task, (uint32_t)ANC_GRAB);
        t0 = __shfl_sync(0xffffffffu, t0, 0);
        if (t0 >= n_tasks) break;
        const int nt = (int)min((uint32_t)ANC_GRAB, n_tasks - t0);
        __syncwarp();  // the previous grab's descriptors are no longer read
        if (lane < nt) sdesc[lane] = desc[t0 + lane];
        __syncwarp();
        auto first_batch = [&](const seed_t *q, int ns, seed_t (&sdn)[PJ]) {
            if constexpr (NARROW)
                load_first_batch_narrow(q, ns, lane, sdn);
            else
                load_first_batch(q, ns, lane, sdn);
        };
        seed_t sdn[PJ];
        first_batch(reinterpret_cast<const seed_t *>(db.seeds + sdesc[0].seed_idx), (int)sdesc[0].nseeds, sdn);
        for (int k = 0; k < nt; k++) {
            // descriptor fields come from shared memory (broadcast reads) where they are used: nothing is held in
            // registers across the grab
            const TaskDesc &d = sdesc[k];
            const int kn = k + 1 < nt ? k + 1 : k;
            const int nseeds = (int)d.nseeds, ns_next = k + 1 < nt ? (int)sdesc[kn].nseeds : 0;
            const seed_t *qs = reinterpret_cast<const seed_t *>(db.seeds + d.seed_idx);
            const seed_t *qs_next = reinterpret_cast<const seed_t *>(db.seeds + sdesc[kn].seed_idx);
            int n = 0;
            if (nseeds > 0) {
                const uint64_t *T = db.tab + d.tab_idx;
                uint64_t *anc = anc_all + slab_base(t0 + k);  // entry i of the task at anc[slab_off(i)]
                // optimistic pass with the full multiplicity cap; if the chunk overflows MAXA, halve the cap
                // until it fits (oracle rule; rare)
                int mult = prm.max_mult;
                for (;;) {
                    if constexpr (NARROW)
                        n = emit_anchors_narrow(qs, nseeds, d.cstart, T, d.nb, mult, prm.max_mult, MAXA, stage, anc, lane, sdn,
                                                qs_next, ns_next);
                    else
                        n = emit_anchors(qs, nseeds, d.cstart, T, d.nb, mult, prm.max_mult, MAXA, stage, anc, lane, sdn, qs_next,
                                         ns_next);
                    if (n <= MAXA || mult == 1) break;
                    mult >>= 1;
                    first_batch(qs, nseeds, sdn);
                }
                if (n > MAXA || n < prm.min_anchors) n = 0;
            } else
                first_batch(qs_next, ns_next, sdn);
            if (lane == 0) task_n[t0 + k] = (uint16_t)n;
            __syncwarp();
        }
    }
}

// ---- K4b: chaining DP, one THREAD per task.
//   Q = q_rel + (rev << 20) + 1: other strand relation => more than band apart, no extra test;
//       the +1 makes (Qi - Q[j]) == dq - 1, so one unsigned compare checks 0 < dq <= band
//   D = R - q with R = rev ? -ref_pos : ref_pos: gap = |D_i - D_j|, d_ref = (D_i - D_j) + dq
//   F = f + anchor_score (0 = empty slot: it can never beat `best`, which starts at anchor_score)
// Colinear anchors (the usual case) chain onto one of the two nearest predecessors with a score no other one can
// reach.  So only those two live in registers (FR = F << 17 | root << 9 | cnt, the ring word, is carried packed: the
// register a shared-memory store reads stays live for two more anchors, so the store never holds the next write to it
// back -- ncu, round 2: those write-after-read waits and the MIO queue were 20 % of the kernel's stall samples with
// three ring stores per anchor); the 16-deep look-back window is a ring of (D, FR) in shared memory, written once per
// anchor and read only on the two rare paths: the bound rebuild and the full scan (which fetches Q from the anchors).
//
// Short cut.  Mx bounds what predecessors beyond the nearest two can offer: the largest F among those whose diagonal
// lies within max_gap + DIAG_SLACK of Dref, where Dref follows this task's current diagonal to within DIAG_SLACK.
// An anchor further off than that is out of max_gap for this one, and one inside offers F - gap <= Mx: if
// Mx <= best nothing replaces `best` (a later predecessor only wins with a strictly larger candidate) -- the same
// result as the full scan.  (Two nearest, not one: FracMinHash samples the same 1/125 of k-mer space in both
// genomes, so ~1.7 % of a pair's anchors are chance matches on a random diagonal; one sits between two anchors of a
// chain and the one after it must reach over it.)  An anchor off the current diagonal (`jump`) needs its own bound
// m2 = max F over the window within reach of ITS diagonal.  `off` keeps one bit per window entry: set iff that
// anchor was off Dref's diagonal when it entered.  If no entry beyond the nearest two is off and the anchor is more
// than max_gap + 2 DIAG_SLACK from Dref, every such entry is out of its reach: m2 is empty without looking (chance
// anchors, and the first anchor after a contig end or rearrangement).  Otherwise the ring is read (rare).  The
// diagonal is adopted as the new Dref only when the previous anchor lies on it too (contig end, indel,
// rearrangement -- not a chance anchor), so the old chain's high scores neither keep the short cut off for the next
// 16 anchors nor does one stray anchor derail it.  Stale entries that have left the window only make Mx too large
// (a missed short cut).
template <bool WIDE>
__global__ void __launch_bounds__(DP_THREADS, 8)
chain_kernel(AniParams prm, uint32_t n_tasks, const uint64_t *__restrict__ anc_all, const uint16_t *__restrict__ task_n,
             uint32_t *__restrict__ res_all, const TaskDesc *__restrict__ desc, Cand *__restrict__ cands,
             uint8_t *__restrict__ task_ncand, uint32_t *__restrict__ slow_list /* [0] count, then task ids */) {
    const uint32_t t = blockIdx.x * DP_THREADS + threadIdx.x;
    const int my_n = t < n_tasks ? (int)task_n[t] : 0;
    const int w_n = (int)__reduce_max_sync(0xffffffffu, (unsigned)my_n);
    if (w_n == 0) return;
    constexpr int UNR = DP_UNR;
    static_assert(UNR == 4 && MAXA % UNR == 0 && LB % UNR == 0, "anchors are fetched one 32-byte sector at a time");
    // Diagonals of opposite strands are up to 2^32 apart.  When every padded position of the database is below
    // 2^30 - 2^21 (any bacterial set) their differences fit an int and the diagonal tests are 32-bit (WIDE = false).
    using diff_t = typename std::conditional<WIDE, long long, int>::type;
    auto adiff = [](int a, int b) {
        const diff_t d = (diff_t)a - (diff_t)b;
        return d < 0 ? -d : d;
    };
    // The look-back window beyond the two nearest predecessors: diagonal and packed (F, root, cnt) per entry, a ring in
    // shared memory ([slot][thread]: conflict-free, slot = anchor index & 15).  The query coordinate is not kept: the
    // only path that wants it (the full scan, ~0.6 % of the steps) re-reads it from the anchor array.
    // Rows are padded by one word: the two uncommon paths read one task's COLUMN with 14 lanes at once (below), and rows
    // DP_THREADS words apart would all fall into one bank.
    constexpr int RS = DP_THREADS + 1;  // ring row stride in words
    __shared__ int ringD[LB * RS];
    __shared__ uint32_t ringFR[LB * RS];  // F << 17 | root << 9 | cnt  (0 = empty)
    __shared__ uint32_t tb_s[ENDS_K][DP_THREADS];  // dynamic indexing without local memory; column per thread
    int *const rd = &ringD[threadIdx.x];
    uint32_t *const rf = &ringFR[threadIdx.x];
    const int lane = threadIdx.x & 31;
    const int *const rd_w = &ringD[threadIdx.x & ~31u];      // this warp's 32 columns: lane L's entry d at [slot * RS + L]
    const uint32_t *const rf_w = &ringFR[threadIdx.x & ~31u];
#pragma unroll
    for (int u = 0; u < LB; u++) rf[u * RS] = 0;
    int Q1 = 0, D1 = 0, Q2 = 0, D2 = 0;  // nearest, second nearest predecessor
    uint32_t FR1 = 0, FR2 = 0;           // their ring words: (f + anchor_score) << 17 | root << 9 | cnt, 0 = none
    const uint32_t tt = t < n_tasks ? t : n_tasks - 1;  // idle lanes read a valid slab and write nothing
    const uint64_t *ap = anc_all + slab_base(tt);  // entry i at ap[slab_off(i)]
    uint32_t *rp = res_all + slab_base(tt);
    const unsigned band = (unsigned)prm.band_bp;
    // chain ends, tracked on the fly: per DP tree (root) the best qualifying end as
    //   (f << 16) | (255 - i) << 8 | root   -- max over a tree = highest score, ties lowest index.
    // Anchors of a tree arrive mostly back to back, so the tree in progress sits in (cur_root, cur_e) and the
    // table of finished trees is touched only when the root changes.  More than ENDS_K qualifying trees in one
    // chunk (rare) hands the task to ends_kernel.  Valid because min_score > (min_anchors - 1) * anchor_score
    // (checked at context creation): an end that reaches min_score has min_anchors anchors, and if the tree's
    // best end does not qualify nothing in the tree does.
    uint32_t *const tb = &tb_s[0][threadIdx.x];
#pragma unroll
    for (int k = 0; k < ENDS_K; k++) tb[k * DP_THREADS] = 0;
    uint32_t cur_root = 0xffffffffu, cur_e = 0;
    bool slow = false;
    auto flush = [&](uint32_t e) {  // kept small on purpose: it is inlined once per unrolled anchor (I-cache)
        if (e == 0) return;
        int k = 0;
#pragma unroll 1
        for (; k < ENDS_K; k++) {  // entries fill front to back and never leave: first empty-or-same-root slot
            const uint32_t v = tb[k * DP_THREADS];
            if (v == 0 || ((v ^ e) & 0xffu) == 0) {
                tb[k * DP_THREADS] = v > e ? v : e;
                break;
            }
        }
        if (k == ENDS_K) slow = true;
    };
    int Mx = 0, Dref = 0;
    uint32_t off = 0;  // bit d: the d-th previous anchor (0 = nearest) is live and off Dref's diagonal
    const int diag_lim = prm.max_gap + DIAG_SLACK;
    // four anchors = one 32-byte sector = one 256-bit load (the slabs are 2 KB apart: nothing to coalesce across lanes)
    auto load4 = [&](int i, uint64_t (&v)[UNR]) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
                     : "=l"(v[0]), "=l"(v[1]), "=l"(v[2]), "=l"(v[3]) : "l"(ap + slab_off((uint32_t)i)));
    };
    uint64_t vnext[UNR];
    load4(0, vnext);
    for (int i0 = 0; i0 < w_n; i0 += UNR) {
        uint64_t av[UNR];
#pragma unroll
        for (int x = 0; x < UNR; x++) av[x] = vnext[x];
        if (i0 + UNR < MAXA) load4(i0 + UNR, vnext);  // next iteration's anchors
        // The body is unrolled DP_BODY times (2), not UNR: at four copies the loop is 24 KB of code and 12 % of the
        // kernel's stall samples were instruction fetches (ncu, round 2); the two halves of a group share one copy.
#pragma unroll 1
        for (int h = 0; h < UNR / DP_BODY; h++) {
        const int ring0 = ((i0 + DP_BODY * h) & (LB - 1)) * RS;  // slot of this half's first anchor
        uint32_t outp[DP_BODY];
#pragma unroll
        for (int x = 0; x < DP_BODY; x++) {
            const uint64_t a = av[x];
            const int rev = (int)an_rev(a);
            const int qi = (int)an_q(a) + (rev << 20);
            const int Ri = rev ? -(int)an_r(a) : (int)an_r(a);
            const int Di = Ri - qi;
            const int i = i0 + DP_BODY * h + x;
            int best = prm.anchor_score;
            uint32_t brc = (uint32_t)i << 9;  // own root, cnt 0 (+1 below)
            const bool live = i < my_n;
            auto relax = [&](int Qj, int Dj, uint32_t FRj) {
                const int dq1 = qi - Qj;  // dq - 1
                const int dd = Di - Dj;
                const int dr1 = dd + dq1;  // d_ref - 1
                const int gap = dd < 0 ? -dd : dd;
                const int cand = (int)(FRj >> 17) - gap;
                if ((unsigned)dq1 < band && dr1 >= 0 && gap <= prm.max_gap && cand > best) {
                    best = cand;
                    brc = FRj & 0x1ffffu;
                }
            };
            relax(Q1, D1, FR1);  // the nearest predecessor: ties keep it
            relax(Q2, D2, FR2);
            const diff_t dj = adiff(Di, Dref);
            bool jump = live && dj > DIAG_SLACK;
            bool settled = !live || Mx <= best;
            if (__any_sync(0xffffffffu, jump)) {
                const diff_t dp = adiff(Di, D1);
                // A far jump leaves every entry on Dref's diagonal (`off` bit clear: within DIAG_SLACK of Dref) out of
                // its reach and off its own diagonal, without looking; only the entries flagged in `off` are read.
                const bool far = dj > diag_lim + DIAG_SLACK;
                const bool quick = far && (off >> 2) == 0;
                const uint32_t window = 0xfffcu & ((1u << (i < LB ? i : LB)) - 1u);  // anchors i-3 .. i-16 that exist (all live)
                int m2 = 0;
                uint32_t offn = far ? window & ~off : 0u;  // `off` relative to this anchor's diagonal, beyond the nearest two
                // The lanes that must look at their ring (a near jump, or a far one with flagged entries) are served
                // one after the other by the whole warp: lane d reads entry d of that task's column, one max-reduction
                // and one ballot give (m2, offn).  A per-lane loop here ran 14 iterations with one lane active --
                // on genomes with repeat families (multi-hit seeds put several diagonals into one window) 19 % of the
                // warp-steps did, and chain_kernel took 17.6 ms per batch instead of 3.9 (ncu, config3r).
                const uint32_t my_todo = (jump && !quick) ? (far ? window & off : window) : 0u;
                for (unsigned need = __ballot_sync(0xffffffffu, my_todo != 0u); need; need &= need - 1) {
                    const int L = __ffs((int)need) - 1;
                    const int DiL = __shfl_sync(0xffffffffu, Di, L);
                    const uint32_t todoL = __shfl_sync(0xffffffffu, my_todo, L);
                    int f_in = 0;
                    bool off_in = false;
                    if ((todoL >> lane) & 1u) {  // lane = d, 2 <= d < LB
                        const int sl = ((i - 1 - lane) & (LB - 1)) * RS + L;
                        const diff_t dd = adiff(rd_w[sl], DiL);
                        if (dd <= diag_lim) f_in = (int)(rf_w[sl] >> 17);
                        off_in = dd > DIAG_SLACK;
                    }
                    const int m2L = (int)__reduce_max_sync(0xffffffffu, (unsigned)f_in);
                    const unsigned offL = __ballot_sync(0xffffffffu, off_in);
                    if (lane == L) {
                        m2 = m2L;
                        offn |= offL;
                    }
                }
                if (jump) {
                    settled = m2 <= best;  // quick: m2 = 0
                    if (dp <= DIAG_SLACK) {  // the previous anchor is on this diagonal too: follow it
                        Mx = m2;
                        Dref = Di;
                        off = offn | ((FR2 != 0 && adiff(D2, Di) > DIAG_SLACK) ? 2u : 0u);
                        jump = false;
                    }
                }
            }
            // Full scan of the window for the lanes the short cut could not settle, again one lane at a time with the
            // warp's help: lane d relaxes against entry d (its query coordinate comes from the anchor array: the 14
            // anchors are consecutive, one or two lines), the best candidate wins by one max-reduction on
            // (cand << 4 | 15 - d): the largest candidate, ties to the nearest -- what the sequential scan gives.
            for (unsigned need = __ballot_sync(0xffffffffu, !settled); need; need &= need - 1) {
                const int L = __ffs((int)need) - 1;
                const int DiL = __shfl_sync(0xffffffffu, Di, L), qiL = __shfl_sync(0xffffffffu, qi, L);
                const int bestL = __shfl_sync(0xffffffffu, best, L);
                const uint32_t ttL = __shfl_sync(0xffffffffu, tt, L);
                uint32_t fr = 0, key = 0;
                if (lane >= 2 && lane < LB && lane <= i - 1) {
                    const int sl = ((i - 1 - lane) & (LB - 1)) * RS + L;
                    fr = rf_w[sl];
                    if (fr) {
                        const uint32_t lo = __ldcg(reinterpret_cast<const uint32_t *>(
                            anc_all + slab_base(ttL) + slab_off((uint32_t)(i - 1 - lane))));
                        const int Qj = (int)((lo >> 17) & 0x7fffu) + (int)(((lo >> 16) & 1u) << 20) + 1;
                        const int dq1 = qiL - Qj, dd = DiL - rd_w[sl], dr1 = dd + dq1;
                        const int gap = dd < 0 ? -dd : dd;
                        const int cand = (int)(fr >> 17) - gap;
                        if ((unsigned)dq1 < band && dr1 >= 0 && gap <= prm.max_gap && cand > bestL)
                            key = ((uint32_t)cand << 4) | (uint32_t)(LB - 1 - lane);
                    }
                }
                const uint32_t kmax = __reduce_max_sync(0xffffffffu, key);
                const uint32_t frs = __shfl_sync(0xffffffffu, fr, LB - 1 - (int)(kmax & 15u));
                if (lane == L && kmax) {
                    best = (int)(kmax >> 4);
                    brc = frs & 0x1ffffu;
                }
            }
            // the second nearest predecessor is beyond the nearest two of the next anchor
            Mx = max(Mx, adiff(D2, Dref) <= diag_lim ? (int)(FR2 >> 17) : 0);
            const uint32_t rci = brc + 1;
            outp[x] = ((uint32_t)best << 17) | rci;
            if (live && best >= prm.min_score && (int)(rci & 0x1ffu) >= prm.min_anchors) {
                const uint32_t root = rci >> 9;
                const uint32_t e = ((uint32_t)best << 16) | ((uint32_t)(MAXA - 1 - i) << 8) | root;
                if (root == cur_root)
                    cur_e = cur_e > e ? cur_e : e;
                else {
                    flush(cur_e);
                    cur_root = root;
                    cur_e = e;
                }
            }
            Q2 = Q1, D2 = D1, FR2 = FR1;
            Q1 = qi + 1, D1 = Di, FR1 = live ? outp[x] + ((uint32_t)prm.anchor_score << 17) : 0u;
            rd[ring0 + x * RS] = D1;
            rf[ring0 + x * RS] = FR1;
            off = ((off << 1) | (jump ? 1u : 0u)) & 0xffffu;
        }
        if (i0 + DP_BODY * h < my_n) {
            if constexpr (DP_BODY == 4)
                __stcg(reinterpret_cast<uint4 *>(rp + slab_off((uint32_t)i0)), make_uint4(outp[0], outp[1], outp[2], outp[3]));
            else
                __stcg(reinterpret_cast<uint2 *>(rp + slab_off((uint32_t)(i0 + DP_BODY * h))), make_uint2(outp[0], outp[1]));
        }
        if constexpr (DP_BODY == 2) {
            av[0] = av[2];
            av[1] = av[3];
        }
        }
    }
    // ---- the chunk's top candidates, by (score desc, q0, r0), into the task's slots
    if (my_n == 0) return;
    flush(cur_e);
    if (slow) {
        slow_list[1 + atomicAdd(&slow_list[0], 1u)] = t;
        return;
    }
    uint64_t key[ENDS_K];
    int m = 0;
#pragma unroll
    for (int k = 0; k < ENDS_K; k++) {
        key[k] = ~0ull;
        const uint32_t e = tb[k * DP_THREADS];
        if (e) {
            const uint64_t ar = __ldcg(ap + slab_off(e & 0xffu));
            const uint64_t ae = __ldcg(ap + slab_off(MAXA - 1 - ((e >> 8) & 0xffu)));
            const uint32_t r0 = an_r(ar) < an_r(ae) ? an_r(ar) : an_r(ae);
            key[k] = ((uint64_t)(8191u - (e >> 16)) << 47) | ((uint64_t)an_q(ar) << 32) | (uint64_t)r0;
            m++;
        }
    }
    const TaskDesc d = desc[t];
    const int n_out = m < prm.max_chunk_chains ? m : prm.max_chunk_chains;
    for (int ord = 0; ord < n_out; ord++) {
        int bk = 0;
        uint64_t bkey = key[0];
#pragma unroll
        for (int k = 1; k < ENDS_K; k++)
            if (key[k] < bkey) {
                bkey = key[k];
                bk = k;
            }
#pragma unroll
        for (int k = 0; k < ENDS_K; k++)
            if (k == bk) key[k] = ~0ull;
        const uint32_t e = tb[bk * DP_THREADS];
        const int iend = MAXA - 1 - (int)((e >> 8) & 0xffu);
        const uint64_t ar = __ldcg(ap + slab_off(e & 0xffu)), ae = __ldcg(ap + slab_off((uint32_t)iend));
        const uint32_t x = __ldcg(rp + slab_off((uint32_t)iend));  // written above by this thread
        Cand c;
        c.q0 = d.cstart + an_q(ar);
        c.q1 = d.cstart + an_q(ae);
        c.r0 = an_r(ar) < an_r(ae) ? an_r(ar) : an_r(ae);
        c.r1 = an_r(ar) < an_r(ae) ? an_r(ae) : an_r(ar);
        c.chunk = d.ch;
        c.score = (uint16_t)(e >> 16);
        c.n_anchors = (uint16_t)rs_cnt(x);
        c.n_seeds = (uint16_t)(an_sidx(ae) - an_sidx(ar) + 1);
        c.ordinal = (uint8_t)ord;
        c.rev = (uint8_t)an_rev(ae);
        c.pad = 0;
        cands[(size_t)t * SLOTS + ord] = c;
    }
    if (n_out) task_ncand[t] = (uint8_t)n_out;
}

// ---- K4c: chain ends (fallback for chunks with more than ENDS_K qualifying trees).  One warp per task: best end of every DP tree (ties: lowest index) with
// >= min_anchors / min_score; the chunk's top `max_chunk_chains` by (score, q0, r0) go to the task's
// fixed candidate slots.
__global__ void __launch_bounds__(END_THREADS)
ends_kernel(AniParams prm, uint32_t n_tasks, const uint64_t *__restrict__ anc_all, const uint32_t *__restrict__ res_all,
            const uint16_t *__restrict__ task_n, const TaskDesc *__restrict__ desc, const uint32_t *__restrict__ slow_list,
            Cand *__restrict__ cands, uint8_t *__restrict__ task_ncand) {
    __shared__ uint32_t bor_all[END_THREADS / 32][MAXA];
    __shared__ __align__(16) uint32_t lst_all[END_THREADS / 32][SLOTS * 8 + SLOTS * 2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *bor = bor_all[warp];
    const uint32_t warps_total = gridDim.x * (END_THREADS / 32);
    const uint32_t n_slow = slow_list[0];  // the tasks chain_kernel could not finish itself (usually none)
    for (uint32_t k = blockIdx.x * (END_THREADS / 32) + warp; k < n_slow; k += warps_total) {
        const uint32_t t = slow_list[1 + k];
        const int n = task_n[t];
        if (n == 0) continue;
        const uint32_t ch_k = desc[t].ch, cstart_k = desc[t].cstart;
        const uint64_t *anc = anc_all + slab_base(t);  // entry i at [slab_off(i)]
        const uint32_t *res = res_all + slab_base(t);
        uint32_t xs[MAXA / 32];
#pragma unroll
        for (int u = 0; u < MAXA / 32; u++) {
            const int i = lane + 32 * u;
            xs[u] = i < n ? __ldcg(res + slab_off((uint32_t)i)) : 0u;
            if (i < n) bor[i] = 0;
        }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < MAXA / 32; u++) {
            const int i = lane + 32 * u;
            if (i < n) atomicMax(&bor[rs_root(xs[u])], (rs_f(xs[u]) << 8) | (uint32_t)(MAXA - 1 - i));
        }
        __syncwarp();
        uint32_t mine = 0;  // bit u <-> i = lane + 32 u
#pragma unroll
        for (int u = 0; u < MAXA / 32; u++) {
            const int i = lane + 32 * u;
            const uint32_t x = xs[u];
            if (i < n && bor[rs_root(x)] == ((rs_f(x) << 8) | (uint32_t)(MAXA - 1 - i)) &&
                (int)rs_cnt(x) >= prm.min_anchors && (int)rs_f(x) >= prm.min_score)
                mine |= 1u << u;
        }
        __syncwarp();
        const int my_cnt = __popc(mine);
        const int total = (int)__reduce_add_sync(0xffffffffu, (unsigned)my_cnt);
        if (total == 0) continue;
        if (total <= prm.max_chunk_chains) {
            // common case: every qualifying end becomes a candidate.  All lanes fetch their ends'
            // anchors at once, publish (candidate, key) to shared memory, then `total` lanes rank the
            // keys for the ordinals.
            int pre = my_cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, pre, d);
                if (lane >= d) pre += u;
            }
            pre -= my_cnt;
            Cand *lst = reinterpret_cast<Cand *>(lst_all[warp]);                  // [SLOTS]
            uint64_t *lkey = reinterpret_cast<uint64_t *>(lst_all[warp] + SLOTS * 8);  // [SLOTS]
#pragma unroll
            for (int u = 0; u < MAXA / 32; u++) {
                if ((mine >> u) & 1u) {
                    const int i = lane + 32 * u;
                    const uint32_t x = xs[u];
                    const uint64_t ar = __ldcg(anc + slab_off(rs_root(x))), ae = __ldcg(anc + slab_off((uint32_t)i));
                    Cand c;
                    c.q0 = cstart_k + an_q(ar);
                    c.q1 = cstart_k + an_q(ae);
                    c.r0 = an_r(ar) < an_r(ae) ? an_r(ar) : an_r(ae);
                    c.r1 = an_r(ar) < an_r(ae) ? an_r(ae) : an_r(ar);
                    c.chunk = ch_k;
                    c.score = (uint16_t)rs_f(x);
                    c.n_anchors = (uint16_t)rs_cnt(x);
                    c.n_seeds = (uint16_t)(an_sidx(ae) - an_sidx(ar) + 1);
                    c.ordinal = 0;
                    c.rev = (uint8_t)an_rev(ae);
                    c.pad = 0;
                    lst[pre] = c;
                    lkey[pre] = ((uint64_t)(8191u - rs_f(x)) << 47) | ((uint64_t)an_q(ar) << 32) | (uint64_t)c.r0;
                    pre++;
                }
            }
            __syncwarp();
            if (lane < total) {
                const uint64_t key = lkey[lane];
                int ord = 0;
                for (int j = 0; j < total; j++) ord += lkey[j] < key;  // keys are unique
                Cand c = lst[lane];
                c.ordinal = (uint8_t)ord;
                cands[(size_t)t * SLOTS + ord] = c;
            }
            if (lane == 0) task_ncand[t] = (uint8_t)total;
            __syncwarp();
            continue;
        }
        // rare: more qualifying ends than slots -> take the best max_chunk_chains, one per round
        int n_out = 0;
        for (int rnd = 0; rnd < prm.max_chunk_chains; rnd++) {
            uint64_t bk = ~0ull;
            int bi = -1;
            for (uint32_t mm = mine; mm; mm &= mm - 1) {
                const int u = __ffs(mm) - 1, i = lane + 32 * u;
                const uint32_t x = __ldcg(res + slab_off((uint32_t)i));
                const uint64_t ar = __ldcg(anc + slab_off(rs_root(x))), ae = __ldcg(anc + slab_off((uint32_t)i));
                const uint32_t r0 = an_r(ar) < an_r(ae) ? an_r(ar) : an_r(ae);
                const uint64_t key = ((uint64_t)(8191u - rs_f(x)) << 47) | ((uint64_t)an_q(ar) << 32) | (uint64_t)r0;
                if (key < bk) {
                    bk = key;
                    bi = i;
                }
            }
            const uint32_t khi = __reduce_min_sync(0xffffffffu, (uint32_t)(bk >> 32));
            if (khi == 0xffffffffu) break;  // no candidate left
            const uint32_t klo = __reduce_min_sync(0xffffffffu, (uint32_t)(bk >> 32) == khi ? (uint32_t)bk : 0xffffffffu);
            if (bk == (((uint64_t)khi << 32) | klo)) {  // keys are unique: exactly one lane
                mine &= ~(1u << ((bi - lane) >> 5));
                const uint32_t x = __ldcg(res + slab_off((uint32_t)bi));
                const uint64_t ar = __ldcg(anc + slab_off(rs_root(x))), ae = __ldcg(anc + slab_off((uint32_t)bi));
                Cand c;
                c.q0 = cstart_k + an_q(ar);
                c.q1 = cstart_k + an_q(ae);
                c.r0 = an_r(ar) < an_r(ae) ? an_r(ar) : an_r(ae);
                c.r1 = an_r(ar) < an_r(ae) ? an_r(ae) : an_r(ar);
                c.chunk = ch_k;
                c.score = (uint16_t)rs_f(x);
                c.n_anchors = (uint16_t)rs_cnt(x);
                c.n_seeds = (uint16_t)(an_sidx(ae) - an_sidx(ar) + 1);
                c.ordinal = (uint8_t)n_out;
                c.rev = (uint8_t)an_rev(ae);
                c.pad = 0;
                cands[(size_t)t * SLOTS + n_out] = c;
            }
            n_out++;
        }
        if (lane == 0 && n_out) task_ncand[t] = (uint8_t)n_out;
        __syncwarp();
    }
}


// A chain as the selection sees it: one 32-byte record in its PAIR's list (the pair's chunks' candidates back to back
// in no particular order), with everything the result needs precomputed -- the finalize kernels touch no other table.
struct __align__(16) PCand {
    uint32_t q0, q1, r0, r1;
    uint16_t score, n_anchors, n_seeds, ext;  // ext: bases the clipped extension adds to both spans
    uint32_t key2;                            // chunk << 4 | ordinal: rank among equal scores
    uint32_t pad;
};
static_assert(sizeof(PCand) == 32, "pcand size");

// Clipped extension of an accepted chain's spans, left + right (the spans themselves are q1-q0+k and r1-r0+k).
__device__ __forceinline__ uint32_t cand_ext(const DbView &db, const AniParams &prm, const Cand &c, uint32_t choff,
                                             uint32_t rcoff, int nrc) {
    const long long e = prm.span_ext, k1 = K_SEED - 1;
    const long long cs = db.chunk_start[choff + c.chunk], ce = cs + db.chunk_len[choff + c.chunk] - 1;
    int lo = 0, hi = nrc - 1;  // reference contig holding r0
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (db.ctg_pstart[rcoff + mid] <= c.r0)
            lo = mid;
        else
            hi = mid - 1;
    }
    const long long rs = db.ctg_pstart[rcoff + lo], re = rs + db.ctg_len[rcoff + lo] - 1;
    const long long a0 = (long long)c.q0 - k1, a1 = c.q1, b0 = (long long)c.r0 - k1, b1 = c.r1;
    const long long room_ql = a0 - cs, room_qr = ce - a1, room_rlo = b0 - rs, room_rhi = re - b1;
    // an extension stops where either genome runs out; a reverse chain's left query end faces the reference's high end
    long long el = c.rev ? room_rhi : room_rlo, er = c.rev ? room_rlo : room_rhi;
    el = el < room_ql ? el : room_ql;
    er = er < room_qr ? er : room_qr;
    el = el < e ? el : e;
    er = er < e ? er : e;
    el = el < 0 ? 0 : el;
    er = er < 0 ? 0 : er;
    return (uint32_t)(el + er);
}

// One thread per task: its candidates (chain_kernel / ends_kernel left them in the task's slots) move to the batch's
// compact list at cand_off[t] (exclusive scan of the tasks' candidate counts): a pair's candidates are contiguous, in
// (chunk, ordinal) order, and cand_off brackets them.  The extension is worked out here, at full occupancy -- the
// contig search is a chain of dependent loads that a warp-per-pair kernel cannot hide.
__global__ void cand_pack_kernel(DbView db, AniParams prm, const PairInfo *__restrict__ info, uint32_t n_tasks,
                                 const uint32_t *__restrict__ task_pair, const uint8_t *__restrict__ task_ncand,
                                 const uint32_t *__restrict__ cand_off, const Cand *__restrict__ gcands,
                                 PCand *__restrict__ pcands) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tasks) return;
    const uint32_t c = task_ncand[t];
    if (c == 0) return;
    const PairInfo pi = info[task_pair[t]];
    const uint32_t choff = db.g_chunk_off[pi.q], rcoff = db.g_ctg_off[pi.r];
    const int nrc = (int)(db.g_ctg_off[pi.r + 1] - rcoff);
    PCand *dst = pcands + cand_off[t];
    for (uint32_t x = 0; x < c; x++) {
        const Cand cd = gcands[(size_t)t * SLOTS + x];
        PCand o;
        o.q0 = cd.q0, o.q1 = cd.q1, o.r0 = cd.r0, o.r1 = cd.r1;
        o.score = cd.score, o.n_anchors = cd.n_anchors, o.n_seeds = cd.n_seeds;
        o.ext = (uint16_t)cand_ext(db, prm, cd, choff, rcoff, nrc);
        o.key2 = (cd.chunk << 4) | cd.ordinal;
        o.pad = 0;
        dst[x] = o;
    }
}

// ANI of `a_in` anchors over `s_in` query seeds (both > 0): raw = ratio^(1/k), then the debias substitute.  The one
// place this arithmetic lives: the pooled mean (make_pair_out), the median / robust estimators (est_pick_kernel),
// the --ci bounds (ci_kernel) and --detailed's per-chain ANI (sd_kernel).
// Two steps, so that make_pair_out keeps its order of work (the AF in between): its register allocation is unchanged.
__device__ __forceinline__ double ani_raw_of(int64_t a_in, int64_t s_in) {
    double ratio = (double)a_in / (double)s_in;
    if (ratio > 1.0) ratio = 1.0;
    return pow(ratio, 1.0 / (double)K_SEED);
}
__device__ __forceinline__ double ani_debiased(const AniParams &prm, double raw) {
    const double x = 100.0 * (1.0 - raw);
    double ani = 1.0;
    if (x > 0.0) {
        ani = 1.0 - prm.debias_a * pow(x, prm.debias_g) / 100.0;
        if (ani < 0.0) ani = 0.0;
    }
    return ani > 1.0 ? 1.0 : ani;
}

// The pair's result from the sums over its accepted chains (one thread).
__device__ __forceinline__ PairOut make_pair_out(const DbView &db, const AniParams &prm, const PairInfo &pi, int64_t t_a,
                                                 int64_t t_s, int64_t t_span_q, int64_t t_span_r, int n_acc) {
    PairOut o;
    o.ani = o.ani_raw = -1.0;
    o.af_q = o.af_r = 0.0;
    o.n_anchors = t_a;
    o.n_seeds = t_s;
    o.span_q = t_span_q;
    o.span_r = t_span_r;
    o.n_chains = n_acc;
    o.swapped = (int32_t)pi.swapped;
    // the two end anchors of every chain are anchors by construction: left out of both counts (oracle ora_pair)
    const int64_t a_in = o.n_anchors - 2 * (int64_t)o.n_chains, s_in = o.n_seeds - 2 * (int64_t)o.n_chains;
    if (a_in > 0 && s_in > 0) {
        o.ani_raw = ani_raw_of(a_in, s_in);
        double afq = (double)o.span_q / (double)db.g_total_len[pi.q];
        double afr = (double)o.span_r / (double)db.g_total_len[pi.r];
        o.af_q = afq > 1.0 ? 1.0 : afq;
        o.af_r = afr > 1.0 ? 1.0 : afr;
        o.ani = ani_debiased(prm, o.ani_raw);
    }
    return o;
}

// does the earlier-ranked chain `d` (q0 q1 r0 r1) overlap more than ovl_num/ovl_den of chain `c`'s own length, on the
// query or on the reference?
__device__ __forceinline__ bool chain_blocks(const uint4 &d, const uint4 &c, const AniParams &prm) {
    const long long lq = (long long)c.y - c.x + 1, lr = (long long)c.w - c.z + 1;
    const long long oq = (long long)(c.y < d.y ? c.y : d.y) - (long long)(c.x > d.x ? c.x : d.x) + 1;
    const long long orr = (long long)(c.w < d.w ? c.w : d.w) - (long long)(c.z > d.z ? c.z : d.z) + 1;
    return (oq > 0 && oq * prm.ovl_den > lq * prm.ovl_num) || (orr > 0 && orr * prm.ovl_den > lr * prm.ovl_num);
}

__device__ __forceinline__ double block_sum(double v, double *scratch /* [FIN_THREADS/32] */, int tid) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    __syncthreads();
    if ((tid & 31) == 0) scratch[tid >> 5] = v;
    __syncthreads();
    double r = 0;
    for (int i = 0; i < FIN_THREADS / 32; i++) r += scratch[i];  // fixed order: deterministic
    return r;
}

struct FinCtl {
    int n_cand, unresolved;
    double red[FIN_THREADS / 32];
};

// Selection + ANI/AF, common case: ONE WARP per pair, no block barriers.  Input: the pair's PCand list
// (cand_pack_kernel): records cand_off[t0] .. cand_off[t0 + nch] of pcands, in (chunk, ordinal) order.
//   A chain can only be blocked by a chain it TOUCHES (on the query or on the reference), and almost none touch:
//   query : chunks are disjoint on the query, so only the (<= SLOTS) chains of one chunk can touch there -- they are
//           neighbours in the list, each is tested against the earlier ordinals of its chunk (on both axes);
//   ref   : the list is ordered by r0 -- a warp bitonic sort of (r0 << 32 | index) in shared memory, skipped when the
//           list is already in that order (colinear genomes) -- and every chain walks its successors while they start
//           at or before its own end: normally none.
//   Touching chains of which the earlier-RANKED one (score desc, chunk, ordinal) covers more than ovl of the later one
//   go to an edge list; a chain is rejected iff an ACCEPTED earlier-ranked chain blocks it -- rounds over the edge
//   list only.  Then the accepted chains' anchors / seeds / spans are summed (integers) and one thread writes the result.
// Pairs with more than `wcap` candidates or more than FW_EDGES blocking relations are listed for the CTA-per-pair
// kernels below (shared memory up to MAXP candidates, global scratch beyond): no pair is ever dropped or capped.
constexpr int FW_WARPS = 4;     // warps (pairs in flight) per CTA
constexpr int FW_EDGES = 256;   // blocking relations per pair the warp kernel resolves itself
__host__ __device__ constexpr size_t fw_bytes_per_warp(uint32_t wcap /* power of two */) {
    return (size_t)wcap * (8 + 1) + (size_t)FW_EDGES * 4 + 16;
}

__device__ __forceinline__ bool ranks_before(uint32_t score_a, uint32_t key2_a, uint32_t score_b, uint32_t key2_b) {
    return score_a > score_b || (score_a == score_b && key2_a < key2_b);
}

// list entries i and j touch: if one blocks the other, append (earlier-ranked << 16 | later-ranked)
__device__ __forceinline__ void fw_edge(const PCand *__restrict__ list, int i, int j, const AniParams &prm, uint32_t *edges,
                                        uint32_t *n_edges) {
    const uint4 a = __ldcg(reinterpret_cast<const uint4 *>(list + i)), b = __ldcg(reinterpret_cast<const uint4 *>(list + j));
    const uint4 a1 = __ldcg(reinterpret_cast<const uint4 *>(list + i) + 1), b1 = __ldcg(reinterpret_cast<const uint4 *>(list + j) + 1);
    const bool i_first = ranks_before(a1.x & 0xffffu, a1.z, b1.x & 0xffffu, b1.z);
    const bool blocks = i_first ? chain_blocks(a, b, prm) : chain_blocks(b, a, prm);
    if (!blocks) return;
    const uint32_t e = atomicAdd(n_edges, 1u);
    if (e < (uint32_t)FW_EDGES) edges[e] = i_first ? ((uint32_t)i << 16) | (uint32_t)j : ((uint32_t)j << 16) | (uint32_t)i;
}

// ctl: [0] largest candidate count among the listed mid pairs, [1] number of big pairs, [2] number of mid pairs.
// ACC (median / robust, --ci, --detailed): also store every candidate's accepted flag at acc[its pcands index].
template <bool ACC>
__global__ void __launch_bounds__(FW_WARPS * 32)
finalize_warp_kernel(DbView db, AniParams prm, const PairInfo *__restrict__ info, const uint32_t *__restrict__ task_off,
                     uint32_t base, int64_t n_pairs, const PCand *__restrict__ pcands, const uint32_t *__restrict__ cand_off,
                     const uint32_t *__restrict__ perm, PairOut *__restrict__ out, uint32_t wcap, uint32_t *ctl,
                     uint32_t *__restrict__ mid_list, uint32_t *__restrict__ big_list, uint32_t *__restrict__ big_nc,
                     uint8_t *__restrict__ acc) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char *my = smem + (size_t)warp * ((fw_bytes_per_warp(wcap) + 15) & ~(size_t)15);
    uint64_t *key = reinterpret_cast<uint64_t *>(my);                           // [wcap] r0 << 32 | list index
    uint32_t *edges = reinterpret_cast<uint32_t *>(my + (size_t)wcap * 8);      // [FW_EDGES] (earlier rank << 16) | later
    uint32_t *n_edges = edges + FW_EDGES;                                       // [1] (+ 3 pad)
    uint8_t *state = reinterpret_cast<uint8_t *>(n_edges + 4);                  // [wcap] low 2 bits: 0 undecided, 1 accepted, 2 rejected
    const int64_t warps_total = (int64_t)gridDim.x * FW_WARPS;
    for (int64_t p = (int64_t)blockIdx.x * FW_WARPS + warp; p < n_pairs; p += warps_total) {
        const PairInfo pi = info[p];
        const uint32_t t0 = task_off[p] - base;
        const uint32_t c0 = cand_off[t0], nc = cand_off[t0 + pi.nch] - c0;
        if (nc > wcap) {
            if (lane == 0) {
                if (nc <= (uint32_t)MAXP) {
                    atomicMax(&ctl[0], nc);
                    mid_list[atomicAdd(&ctl[2], 1u)] = (uint32_t)p;
                } else {
                    const uint32_t k = atomicAdd(&ctl[1], 1u);
                    big_list[k] = (uint32_t)p;
                    big_nc[k] = nc;
                }
            }
            continue;
        }
        const PCand *list = pcands + c0;
        const int n = (int)nc;
        int m = 32;
        while (m < n) m <<= 1;
        // ---- keys; is the list already ordered by r0?
        bool ordered = true;
        for (int t = lane; t < m; t += 32) {
            uint64_t k = ~0ull;
            if (t < n) {
                const uint32_t r0 = __ldcg(&list[t].r0);
                k = ((uint64_t)r0 << 32) | (uint32_t)t;
                state[t] = 1;
            }
            key[t] = k;
            const uint64_t prev = __shfl_up_sync(0xffffffffu, k, 1);
            if (lane > 0 && prev > k) ordered = false;
        }
        if (lane == 0) *n_edges = 0;
        __syncwarp();
        for (int t = 32 + lane; t < n; t += 32)  // across the rows of 32
            if (lane == 0 && key[t - 1] > key[t]) ordered = false;
        if (!__all_sync(0xffffffffu, ordered)) {
            for (int k = 2; k <= m; k <<= 1)
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int t = lane; t < (m >> 1); t += 32) {
                        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                        const int q = i | j;
                        const bool up = (i & k) == 0;
                        const uint64_t a = key[i], b = key[q];
                        if ((a > b) == up) {
                            key[i] = b;
                            key[q] = a;
                        }
                    }
                    __syncwarp();
                }
        }
        // ---- touching chains: later ordinals of the same chunk (any axis), successors in r0 order (reference)
        for (int t = lane; t < n; t += 32) {
            const uint32_t k2 = __ldcg(&list[t].key2);
            const int ord = (int)(k2 & 15u);
            if (ord) {  // rare
                const uint4 c = __ldcg(reinterpret_cast<const uint4 *>(list + t));
                for (int u = t - ord; u < t; u++) {
                    const uint4 d = __ldcg(reinterpret_cast<const uint4 *>(list + u));
                    if ((d.x <= c.y && c.x <= d.y) || (d.z <= c.w && c.z <= d.w)) fw_edge(list, u, t, prm, edges, n_edges);
                }
            }
        }
        for (int s = lane; s < n; s += 32) {
            const int i = (int)(key[s] & 0xffffu);
            const uint32_t r1 = __ldcg(&list[i].r1);
            for (int u = s + 1; u < n && (uint32_t)(key[u] >> 32) <= r1; u++) {  // rare
                const int j = (int)(key[u] & 0xffffu);
                if ((__ldcg(&list[i].key2) >> 4) != (__ldcg(&list[j].key2) >> 4)) fw_edge(list, i, j, prm, edges, n_edges);
            }
        }
        __syncwarp();
        const uint32_t ne = *n_edges;
        if (ne > (uint32_t)FW_EDGES) {  // rare: the CTA kernel takes the pair
            if (lane == 0) {
                atomicMax(&ctl[0], nc);
                mid_list[atomicAdd(&ctl[2], 1u)] = (uint32_t)p;
            }
            __syncwarp();
            continue;
        }
        if (ne) {
            for (uint32_t e = lane; e < ne; e += 32) state[edges[e] & 0xffffu] = 0;
            __syncwarp();
            // state of a blocked chain: bit 2 = an accepted chain blocks it, bit 3 = an undecided one might
            for (;;) {
                for (uint32_t e = lane; e < ne; e += 32) {
                    const uint32_t lo = edges[e] >> 16, hi = edges[e] & 0xffffu;
                    if ((state[hi] & 3) == 0) {
                        const uint8_t s = state[lo] & 3;
                        if (s == 1) atomicOr(reinterpret_cast<unsigned int *>(state + (hi & ~3u)), 4u << (8 * (hi & 3u)));
                        if (s == 0) atomicOr(reinterpret_cast<unsigned int *>(state + (hi & ~3u)), 8u << (8 * (hi & 3u)));
                    }
                }
                __syncwarp();
                bool open = false;
                for (uint32_t e = lane; e < ne; e += 32) {
                    const uint32_t hi = edges[e] & 0xffffu;
                    const uint8_t s = state[hi];
                    if ((s & 3) == 0) {
                        // several edges may share `hi`: they all compute the same value from the same flags
                        if (s & 4) state[hi] = 2;
                        else if (!(s & 8)) state[hi] = 1;
                        else open = true;
                    }
                }
                __syncwarp();
                if (!__any_sync(0xffffffffu, open)) break;
                for (uint32_t e = lane; e < ne; e += 32) {  // undecided chains start the next round with clean flags
                    const uint32_t hi = edges[e] & 0xffffu;
                    if ((state[hi] & 3) == 0) state[hi] = 0;
                }
                __syncwarp();
            }
        }
        // ---- sums over the accepted chains
        uint32_t s_q = 0, s_r = 0, s_a = 0, s_s = 0, n_acc = 0;  // a lane sums <= wcap/32 spans: far below 2^32
        for (int t = lane; t < n; t += 32) {
            if (ACC) acc[c0 + t] = (state[t] & 3) == 1;
            if ((state[t] & 3) != 1) continue;
            const uint4 w0 = __ldcg(reinterpret_cast<const uint4 *>(list + t));
            const uint2 w1 = __ldcg(reinterpret_cast<const uint2 *>(list + t) + 2);  // score n_anchors | n_seeds ext
            const uint32_t ext = w1.y >> 16;
            s_q += w0.y - w0.x + (uint32_t)K_SEED + ext;
            s_r += w0.w - w0.z + (uint32_t)K_SEED + ext;
            s_a += w1.x >> 16;
            s_s += w1.y & 0xffffu;
            n_acc++;
        }
        unsigned long long t_q = s_q, t_r = s_r;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            t_q += __shfl_down_sync(0xffffffffu, t_q, d);
            t_r += __shfl_down_sync(0xffffffffu, t_r, d);
        }
        s_a = __reduce_add_sync(0xffffffffu, s_a);
        s_s = __reduce_add_sync(0xffffffffu, s_s);
        n_acc = __reduce_add_sync(0xffffffffu, n_acc);
        if (lane == 0) out[perm[p]] = make_pair_out(db, prm, pi, (int64_t)s_a, (int64_t)s_s, (int64_t)t_q, (int64_t)t_r, (int)n_acc);
        __syncwarp();
    }
}

constexpr size_t FIN_BYTES_PER_CAND = sizeof(PCand) + 8 + 1;  // candidate + sort key + state

// sort key of a candidate: score desc, chunk, ordinal within the chunk (= (q0, r0) order), then its slot
//   (8191 - score)(13) << 51 | chunk(23) << 28 | ordinal(4) << 24 | slot(24)
constexpr uint32_t FIN_IDX_MASK = 0xffffffu;
constexpr uint32_t MAX_CHUNKS_PER_GENOME = 1u << 23;

// The pairs finalize_warp_kernel listed: one CTA per listed pair.
// BIG = false: candidates / keys / states in dynamic shared memory sized for `cap` candidates (a power of two >= the
//   largest listed pair): PCand[cap] | u64 key[cap] | u8 state[cap].
// BIG = true: the same three arrays in global scratch at big_off[blockIdx.x] (bytes), capacity big_cap[blockIdx.x].
// ACC: as in finalize_warp_kernel.
template <bool BIG, bool ACC>
__global__ void __launch_bounds__(FIN_THREADS)
finalize_kernel(DbView db, AniParams prm, const PairInfo *__restrict__ info, const uint32_t *__restrict__ task_off,
                uint32_t base, int64_t n_pairs, const PCand *__restrict__ pcands, const uint32_t *__restrict__ cand_off,
                const uint32_t *__restrict__ perm, PairOut *__restrict__ out,
                uint32_t cap, const uint32_t *__restrict__ list, const unsigned long long *__restrict__ big_off,
                const uint32_t *__restrict__ big_cap, unsigned char *__restrict__ big_scratch, uint8_t *__restrict__ acc) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ FinCtl ctl;
    const int tid = threadIdx.x;
    const int64_t p = list[blockIdx.x];
    unsigned char *buf = smem;
    if (BIG) {
        cap = big_cap[blockIdx.x];
        buf = big_scratch + big_off[blockIdx.x];
    }
    if (p >= n_pairs) return;
    const PairInfo pi = info[p];
    const uint32_t t0 = task_off[p] - base;
    const PCand *src = pcands + cand_off[t0];
    const int nc = (int)(cand_off[t0 + pi.nch] - cand_off[t0]);
    PCand *cands = reinterpret_cast<PCand *>(buf);
    uint64_t *skey = reinterpret_cast<uint64_t *>(buf + sizeof(PCand) * (size_t)cap);
    uint8_t *state = buf + (sizeof(PCand) + 8) * (size_t)cap;
    int m = 1;
    while (m < nc) m <<= 1;
    for (int i = tid; i < m; i += FIN_THREADS) {
        if (i < nc) {
            const PCand c = src[i];
            cands[i] = c;
            skey[i] = ((uint64_t)(8191u - c.score) << 51) | ((uint64_t)c.key2 << 24) | (uint64_t)i;
        } else
            skey[i] = ~0ull;
        state[i] = 0;
    }
    __syncthreads();
    for (int k = 2; k <= m; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (m >> 1); t += FIN_THREADS) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int q = i | j;
                const bool up = (i & k) == 0;
                const uint64_t a = skey[i], b = skey[q];
                if ((a > b) == up) {
                    skey[i] = b;
                    skey[q] = a;
                }
            }
            __syncthreads();
        }
    }
    // greedy non-overlap selection, resolved in parallel rounds.
    // state: 0 unknown, 1 accepted, 2 rejected.  The candidate at sorted rank t is accepted iff no
    // ACCEPTED candidate of lower rank overlaps more than ovl_num/ovl_den of ITS length on query or ref.
    for (;;) {
        __syncthreads();
        if (tid == 0) ctl.unresolved = 0;
        __syncthreads();
        // rank t costs t comparisons: give every thread one cheap and one expensive rank (tt, nc-1-tt)
        for (int w0 = tid; 2 * w0 < nc; w0 += FIN_THREADS) {
            for (int side = 0; side < 2; side++) {
                const int t = side ? nc - 1 - w0 : w0;
                if (side && t == w0) break;
                if (state[t]) continue;
                const uint4 cr = *reinterpret_cast<const uint4 *>(&cands[(int)(skey[t] & FIN_IDX_MASK)]);  // q0 q1 r0 r1
                int verdict = 1;
                for (int u = 0; u < t; u++) {
                    const uint4 dr = *reinterpret_cast<const uint4 *>(&cands[(int)(skey[u] & FIN_IDX_MASK)]);
                    // intervals that do not even touch (the usual case) cannot block: two compares each
                    const bool tq = dr.x <= cr.y && cr.x <= dr.y, tr = dr.z <= cr.w && cr.z <= dr.w;
                    if (!tq && !tr) continue;
                    const uint8_t su = ((volatile uint8_t *)state)[u];
                    if (su == 2) continue;
                    if (!chain_blocks(dr, cr, prm)) continue;
                    if (su == 1) {
                        verdict = 2;
                        break;
                    }
                    verdict = 0;  // blocked by an undecided candidate: wait
                }
                if (verdict)
                    ((volatile uint8_t *)state)[t] = (uint8_t)verdict;
                else
                    ctl.unresolved = 1;
            }
        }
        __syncthreads();
        if (!ctl.unresolved) break;
    }
    // accumulate accepted chains: anchors / seeds (pooled), spans with the clipped extension
    int n_acc_local = 0;
    double l_span_q = 0, l_span_r = 0, l_a = 0, l_s = 0;  // exact in double (< 2^53); reduced below, no atomics
    for (int t = tid; t < nc; t += FIN_THREADS) {
        if (ACC) acc[cand_off[t0] + (skey[t] & FIN_IDX_MASK)] = state[t] == 1;
        if (state[t] != 1) continue;
        n_acc_local++;
        const PCand &c = cands[(int)(skey[t] & FIN_IDX_MASK)];
        l_span_q += (double)(c.q1 - c.q0 + (uint32_t)K_SEED + c.ext);
        l_span_r += (double)(c.r1 - c.r0 + (uint32_t)K_SEED + c.ext);
        l_a += (double)c.n_anchors;
        l_s += (double)c.n_seeds;
    }
    const double t_span_q = block_sum(l_span_q, ctl.red, tid), t_span_r = block_sum(l_span_r, ctl.red, tid);
    const double t_a = block_sum(l_a, ctl.red, tid), t_s = block_sum(l_s, ctl.red, tid);
    const double t_acc = block_sum((double)n_acc_local, ctl.red, tid);
    if (tid == 0)
        out[perm[p]] = make_pair_out(db, prm, pi, (int64_t)t_a, (int64_t)t_s, (int64_t)t_span_q, (int64_t)t_span_r, (int)t_acc);
}

// ---- --median / --robust (DESIGN.md section 3): after the finalize kernels, per batch --------------------------------
// est_key_kernel (thread per candidate) -> stable segmented sort of (key, candidate index), one segment per pair ->
// est_pick_kernel (warp per pair).  The mean needs none of it.
//
// key of an accepted chain: (a << 47) / s with a = n_anchors - 2, s = n_seeds - 2 (both < 2^16, so distinct ratios get
// distinct keys and equal ratios equal keys); a rejected chain sorts last.  The sort is stable and a pair's candidates
// are listed in (chunk, ordinal) order, which breaks ties.  seg[p] (p <= n_pairs): first candidate of pair p.
__global__ void est_key_kernel(const PCand *__restrict__ pcands, const uint8_t *__restrict__ acc, uint32_t n_cand,
                               const uint32_t *__restrict__ task_off, uint32_t base, int64_t n_pairs,
                               const uint32_t *__restrict__ cand_off, unsigned long long *__restrict__ key,
                               uint32_t *__restrict__ idx, uint32_t *__restrict__ seg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_cand) {
        unsigned long long k = ~0ull;
        if (acc[i]) {
            const PCand &c = pcands[i];
            k = ((unsigned long long)(c.n_anchors - 2u) << 47) / (unsigned long long)(c.n_seeds - 2u);
        }
        key[i] = k;
        idx[i] = (uint32_t)i;
    }
    if (i <= n_pairs) seg[i] = cand_off[task_off[i] - base];
}

// One warp per pair with an estimate: its accepted chains are the first n_chains of its sorted segment.  W = sum of
// the weights s; C = their inclusive prefix, built 32 chains a round with a warp scan.
//   median: the first chain with 2 C >= W (ballot);  robust: pooled a / s over the chains with 10 C > W and
//   10 (C - s) < 9 W.  Rewrites ani / ani_raw; AF and the counts stay the totals over all accepted chains.
__global__ void __launch_bounds__(FW_WARPS * 32)
est_pick_kernel(AniParams prm, int32_t estimator /* SKB_ANI_MEDIAN or _ROBUST */, int64_t n_pairs, const uint32_t *__restrict__ seg,
                const uint32_t *__restrict__ sorted, const PCand *__restrict__ pcands, const uint32_t *__restrict__ perm,
                PairOut *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * FW_WARPS;
    for (int64_t p = (int64_t)blockIdx.x * FW_WARPS + (threadIdx.x >> 5); p < n_pairs; p += warps_total) {
        PairOut &o = out[perm[p]];
        if (o.ani_raw < 0.0) continue;
        const int n = o.n_chains;
        const long long W = o.n_seeds - 2ll * n;
        const uint32_t *list = sorted + seg[p];
        long long carry = 0, sa = 0, ss = 0;
        for (int r0 = 0; r0 < n; r0 += 32) {
            const int t = r0 + lane;
            long long a = 0, s = 0;
            if (t < n) {
                const uint2 w = __ldg(reinterpret_cast<const uint2 *>(pcands + list[t]) + 2);  // score n_anchors | n_seeds ext
                a = (long long)(w.x >> 16) - 2;
                s = (long long)(w.y & 0xffffu) - 2;
            }
            long long C = s;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const long long y = __shfl_up_sync(0xffffffffu, C, d);
                if (lane >= d) C += y;
            }
            C += carry;
            if (estimator == SKB_ANI_MEDIAN) {
                const unsigned hit = __ballot_sync(0xffffffffu, t < n && 2 * C >= W);
                if (hit) {
                    const int src = __ffs(hit) - 1;
                    sa = __shfl_sync(0xffffffffu, a, src);
                    ss = __shfl_sync(0xffffffffu, s, src);
                    break;
                }
            } else if (t < n && 10 * C > W && 10 * (C - s) < 9 * W) {
                sa += a;
                ss += s;
            }
            carry = __shfl_sync(0xffffffffu, C, 31);
            if (10 * carry >= 9 * W) break;  // every later chain starts at or beyond 9W/10: trimmed (median: found)
        }
        if (estimator != SKB_ANI_MEDIAN) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                sa += __shfl_down_sync(0xffffffffu, sa, d);
                ss += __shfl_down_sync(0xffffffffu, ss, d);
            }
        }
        if (lane == 0) {
            o.ani_raw = ani_raw_of(sa, ss);
            o.ani = ani_debiased(prm, o.ani_raw);
        }
    }
}

// ---- --ci (DESIGN.md section 3): percentile-bootstrap interval of the mean ANI, after the finalize kernels, per batch --
// ci_kernel, one warp per pair with an estimate:
//   1. its accepted chains, in candidate ((chunk, ordinal)) order, go to `chains` at the pair's candidate offset as
//      (a << 16 | s), a = n_anchors - 2, s = n_seeds - 2 (a ballot scan over the accepted flags);
//   2. CI_REPS replicates draw n chains each with replacement (lane per replicate, the last few split over 8 lanes);
//   3. the replicates are ranked by A_b / S_b exactly (128-bit cross products, ties by b: a bitonic sort of their indices
//      in shared memory), and ranks CI_LO and CI_HI become (lo, hi) through the same ratio -> raw -> debiased arithmetic
//      as the ANI.  ci[perm[p]] = (lo, hi) as fractions; (-1, -1) for a pair without an estimate.
// Integers throughout up to the two pow calls: s >= a >= 1 for every chain (min_anchors >= 3, one seed per anchor).
constexpr int CI_REPS = 100, CI_LO = 5, CI_HI = 94;
constexpr int CI_SORT = 128;  // the bitonic network's size (>= CI_REPS)

__device__ __forceinline__ uint64_t ci_mix(uint64_t z) {  // splitmix64 finalizer
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// replicate x sorts after replicate y: A_x / S_x > A_y / S_y, ties by index; indices >= CI_REPS (padding) last
__device__ __forceinline__ bool ci_after(int x, int y, const unsigned long long *ra, const unsigned long long *rs) {
    if (x >= CI_REPS || y >= CI_REPS) return x > y;
    const unsigned long long hx = __umul64hi(ra[x], rs[y]), hy = __umul64hi(ra[y], rs[x]);
    if (hx != hy) return hx > hy;
    const unsigned long long lx = ra[x] * rs[y], ly = ra[y] * rs[x];
    return lx != ly ? lx > ly : x > y;
}

__global__ void __launch_bounds__(FW_WARPS * 32)
ci_kernel(AniParams prm, const PairInfo *__restrict__ info, const uint32_t *__restrict__ task_off, uint32_t base,
          int64_t n_pairs, const PCand *__restrict__ pcands, const uint32_t *__restrict__ cand_off,
          const uint8_t *__restrict__ acc, uint32_t *__restrict__ chains, const uint32_t *__restrict__ perm,
          const PairOut *__restrict__ out, double2 *__restrict__ ci) {
    __shared__ unsigned long long s_a[FW_WARPS][CI_REPS], s_s[FW_WARPS][CI_REPS];
    __shared__ uint8_t s_idx[FW_WARPS][CI_SORT];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long *ra = s_a[warp], *rs = s_s[warp];
    uint8_t *idx = s_idx[warp];
    const int64_t warps_total = (int64_t)gridDim.x * FW_WARPS;
    for (int64_t p = (int64_t)blockIdx.x * FW_WARPS + warp; p < n_pairs; p += warps_total) {
        const uint32_t dst = perm[p];
        const PairOut &o = out[dst];
        if (o.ani_raw < 0.0) {
            if (lane == 0) ci[dst] = make_double2(-1.0, -1.0);
            continue;
        }
        // ---- 1. accepted chains, compacted
        const PairInfo pi = info[p];
        const uint32_t t0 = task_off[p] - base;
        const uint32_t c0 = cand_off[t0], nc = cand_off[t0 + pi.nch] - c0;
        uint32_t *list = chains + c0;
        uint32_t m = 0;
        for (uint32_t r0 = 0; r0 < nc; r0 += 32) {
            const uint32_t t = r0 + lane;
            const bool on = t < nc && __ldg(acc + c0 + t);
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            if (on) {
                const uint2 w = __ldg(reinterpret_cast<const uint2 *>(pcands + c0 + t) + 2);  // score n_anchors | n_seeds ext
                list[m + __popc(bal & ((1u << lane) - 1u))] = (((w.x >> 16) - 2u) << 16) | ((w.y & 0xffffu) - 2u);
            }
            m += __popc(bal);
        }
        __syncwarp();
        // ---- 2. replicates: (A_b, S_b) over n draws j = (mix(seed ^ b << 40 ^ i) * n) >> 64
        const unsigned long long n = (unsigned long long)o.n_chains;  // == m
        const unsigned long long A = (unsigned long long)o.n_anchors - 2 * n, S = (unsigned long long)o.n_seeds - 2 * n;
        const unsigned long long seed = ci_mix(ci_mix(ci_mix(n) ^ A) ^ S);
        constexpr int FULL = CI_REPS / 32 * 32;  // replicates one lane draws alone
        for (int b = lane; b < FULL; b += 32) {
            const unsigned long long rb = seed ^ ((unsigned long long)b << 40);
            unsigned long long sa = 0, ss = 0;
            for (unsigned long long i = 0; i < n; i++) {
                const uint32_t v = list[__umul64hi(ci_mix(rb ^ i), n)];
                sa += v >> 16;
                ss += v & 0xffffu;
            }
            ra[b] = sa;
            rs[b] = ss;
        }
        static_assert(CI_REPS - FULL <= 4, "the remaining replicates take 8 lanes each");
        {
            const int b = FULL + (lane >> 3);
            const unsigned long long rb = seed ^ ((unsigned long long)b << 40);
            unsigned long long sa = 0, ss = 0;
            if (b < CI_REPS)
                for (unsigned long long i = lane & 7; i < n; i += 8) {
                    const uint32_t v = list[__umul64hi(ci_mix(rb ^ i), n)];
                    sa += v >> 16;
                    ss += v & 0xffffu;
                }
#pragma unroll
            for (int d = 4; d > 0; d >>= 1) {
                sa += __shfl_xor_sync(0xffffffffu, sa, d);
                ss += __shfl_xor_sync(0xffffffffu, ss, d);
            }
            if (b < CI_REPS && (lane & 7) == 0) {
                ra[b] = sa;
                rs[b] = ss;
            }
        }
        for (int t = lane; t < CI_SORT; t += 32) idx[t] = (uint8_t)t;
        __syncwarp();
        // ---- 3. rank: bitonic sort of the replicate indices
        for (int k = 2; k <= CI_SORT; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = lane; t < CI_SORT / 2; t += 32) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int q = i | j;
                    const bool up = (i & k) == 0;
                    const int x = idx[i], y = idx[q];
                    if (ci_after(x, y, ra, rs) == up) {
                        idx[i] = (uint8_t)y;
                        idx[q] = (uint8_t)x;
                    }
                }
                __syncwarp();
            }
        if (lane == 0) {
            const int lo = idx[CI_LO], hi = idx[CI_HI];
            ci[dst] = make_double2(ani_debiased(prm, ani_raw_of((int64_t)ra[lo], (int64_t)rs[lo])),
                                   ani_debiased(prm, ani_raw_of((int64_t)ra[hi], (int64_t)rs[hi])));
        }
        __syncwarp();
    }
}

// ---- --detailed (DESIGN.md section 3): spread of the chain identities, after ci_kernel, per batch ------------------
// sd_kernel, one warp per pair with an estimate, over the chain list ci_kernel compacted at the pair's candidate offset
// ((a << 16 | s), n_chains of them, no cap): d_c = the ANI of chain c alone (ratio -> raw -> debiased, as the ANI),
// mu = sum s_c d_c / W, sd = sqrt(sum s_c (d_c - mu)^2 / W), W = sum s_c; two passes (d_c recomputed in the second).
// sd[perm[p]] as a fraction; 0 for a one-chain pair, -1 for a pair without an estimate.
__device__ __forceinline__ double sd_chain_ani(const AniParams &prm, uint32_t v) {
    return ani_debiased(prm, ani_raw_of((int64_t)(v >> 16), (int64_t)(v & 0xffffu)));
}

__global__ void __launch_bounds__(FW_WARPS * 32)
sd_kernel(AniParams prm, const uint32_t *__restrict__ task_off, uint32_t base, int64_t n_pairs,
          const uint32_t *__restrict__ cand_off, const uint32_t *__restrict__ chains, const uint32_t *__restrict__ perm,
          const PairOut *__restrict__ out, double *__restrict__ sd) {
    const int lane = threadIdx.x & 31;
    const int64_t warps_total = (int64_t)gridDim.x * FW_WARPS;
    for (int64_t p = (int64_t)blockIdx.x * FW_WARPS + (threadIdx.x >> 5); p < n_pairs; p += warps_total) {
        const uint32_t dst = perm[p];
        const PairOut &o = out[dst];
        const int n = o.n_chains;
        if (o.ani_raw < 0.0 || n == 1) {
            if (lane == 0) sd[dst] = o.ani_raw < 0.0 ? -1.0 : 0.0;
            continue;
        }
        const uint32_t *list = chains + cand_off[task_off[p] - base];
        const double W = (double)(o.n_seeds - 2ll * n);  // exact: < 2^53
        double m = 0.0;
        for (int t = lane; t < n; t += 32) {
            const uint32_t v = list[t];
            m += (double)(v & 0xffffu) * sd_chain_ani(prm, v);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) m += __shfl_xor_sync(0xffffffffu, m, d);
        const double mu = m / W;
        double q = 0.0;
        for (int t = lane; t < n; t += 32) {
            const uint32_t v = list[t];
            const double e = sd_chain_ani(prm, v) - mu;
            q += (double)(v & 0xffffu) * e * e;
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) q += __shfl_down_sync(0xffffffffu, q, d);
        if (lane == 0) sd[dst] = sqrt(q / W);
    }
}

// K5 -- edge compaction: keep pairs with an estimate and max(AF) >= min_af; percent units.  Order-preserving
// (flag -> exclusive scan -> scatter): the pair list is sorted by (a, b), so the edge list comes out sorted too.
__device__ __forceinline__ bool edge_kept(const PairOut &o, double min_af) {
    const double afa = o.swapped ? o.af_r : o.af_q, afb = o.swapped ? o.af_q : o.af_r;
    return o.ani >= 0.0 && (afa >= min_af || afb >= min_af);
}
__global__ void edge_flag_kernel(const PairOut *__restrict__ po, int64_t n_pairs, double min_af /* fraction */,
                                 uint32_t *__restrict__ flag) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n_pairs) flag[t] = edge_kept(po[t], min_af) ? 1u : 0u;
}
__global__ void edge_scatter_kernel(const unsigned long long *__restrict__ pairs, const PairOut *__restrict__ po,
                                    int64_t n_pairs, const uint32_t *__restrict__ flag, const uint32_t *__restrict__ pos,
                                    skb_edge *__restrict__ edges, unsigned long long *n_edges) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs) return;
    if (t == n_pairs - 1) *n_edges = (unsigned long long)pos[t] + flag[t];
    if (!flag[t]) return;
    const PairOut &o = po[t];
    skb_edge e;
    e.a = (uint32_t)(pairs[t] >> 32);
    e.b = (uint32_t)(pairs[t] & 0xffffffffu);
    e.ani = o.ani * 100.0;
    e.af_a = (o.swapped ? o.af_r : o.af_q) * 100.0;
    e.af_b = (o.swapped ? o.af_q : o.af_r) * 100.0;
    edges[pos[t]] = e;
}
// --ci only: the kept pairs' intervals in edge order, percent (edge_flag_kernel's flags, their scan)
__global__ void edge_ci_scatter_kernel(const double2 *__restrict__ ci, int64_t n_pairs, const uint32_t *__restrict__ flag,
                                       const uint32_t *__restrict__ pos, double2 *__restrict__ edge_ci) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs || !flag[t]) return;
    edge_ci[pos[t]] = make_double2(ci[t].x * 100.0, ci[t].y * 100.0);
}
// --detailed only: the kept pairs' details in edge order (edge_flag_kernel's flags, their scan): the interval as
// edge_ci_scatter_kernel writes it, sd in percent, and the AF numerators picked by `swapped` as edge_scatter_kernel
// picks the AF
__global__ void edge_detail_scatter_kernel(const PairOut *__restrict__ po, const double2 *__restrict__ ci,
                                           const double *__restrict__ sd, int64_t n_pairs, const uint32_t *__restrict__ flag,
                                           const uint32_t *__restrict__ pos, skb_edge_detail *__restrict__ detail) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs || !flag[t]) return;
    const PairOut &o = po[t];
    skb_edge_detail d;
    d.ani_lo = ci[t].x * 100.0;
    d.ani_hi = ci[t].y * 100.0;
    d.sd = sd[t] * 100.0;
    d.covered_a = o.swapped ? o.span_r : o.span_q;
    d.covered_b = o.swapped ? o.span_q : o.span_r;
    d.n_chains = o.n_chains;
    d.pad = 0;
    detail[pos[t]] = d;
}

// bookkeeping: sum over pairs of the query genome's seed count and of the chained anchors (roofline bytes)
__global__ void pair_sums_kernel(const PairInfo *__restrict__ info, const PairOut *__restrict__ po, int64_t n_pairs,
                                 const uint64_t *__restrict__ g_seed_off, unsigned long long *sums /* [2] */) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long sq = 0, an = 0;
    if (t < n_pairs) {
        const uint32_t q = info[t].q;
        sq = g_seed_off[q + 1] - g_seed_off[q];
        an = (unsigned long long)po[t].n_anchors;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        sq += __shfl_down_sync(0xffffffffu, sq, d);
        an += __shfl_down_sync(0xffffffffu, an, d);
    }
    if ((threadIdx.x & 31) == 0 && (sq | an)) {
        atomicAdd(&sums[0], sq);
        atomicAdd(&sums[1], an);
    }
}

}  // namespace skb
