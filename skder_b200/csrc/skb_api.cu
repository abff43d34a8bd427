// C-ABI of libskani_b200.so (include/skani_b200.h): context, device buffers, kernel launches.
// No CPU fallback anywhere: every compute entry point launches the sm_100a kernels or fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <ctime>
#include <cub/cub.cuh>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "skb_ani.cuh"
#include "skb_best_n.cuh"
#include "skb_common.cuh"
#include "skb_index.cuh"
#include "skb_matrix.cuh"
#include "skb_sketch.cuh"
#include "skb_table_blocks.cuh"

using namespace skb;

namespace {

thread_local std::string g_create_error;

struct CudaFail {
    std::string msg;
};

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess)                                                                           \
            throw CudaFail{std::string(#call) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" + \
                           std::to_string(__LINE__) + ")"};                                               \
    } while (0)

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;  // elements
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    // grow to at least n elements, keeping the first `keep` elements
    void reserve(size_t n, size_t keep, cudaStream_t st) {
        if (n <= cap) return;
        size_t ncap = std::max(n, cap + cap / 2);
        T *q = nullptr;
        CK(cudaMalloc(&q, ncap * sizeof(T)));
        if (p && keep) CK(cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, st));
        if (p) {
            CK(cudaStreamSynchronize(st));
            cudaFree(p);
        }
        p = q;
        cap = ncap;
    }
    // device copy of h whose first `from` elements are already in place (from = 0: all of it)
    void upload(const std::vector<T> &h, size_t from, cudaStream_t st) {
        reserve(std::max<size_t>(h.size(), 1), from, st);
        if (h.size() > from)
            CK(cudaMemcpyAsync(p + from, h.data() + from, (h.size() - from) * sizeof(T), cudaMemcpyHostToDevice, st));
    }
};

// Typed view of a persistent, grow-only scratch buffer owned by the context: the steady state of
// every entry point performs no cudaMalloc/cudaFree.
template <typename T>
struct PoolRef {
    DevBuf<unsigned char> &b;
    T *p;
    explicit PoolRef(DevBuf<unsigned char> &buf) : b(buf), p(reinterpret_cast<T *>(buf.p)) {}
    void reserve(size_t n, size_t keep, cudaStream_t st) {
        b.reserve(n * sizeof(T), keep * sizeof(T), st);
        p = reinterpret_cast<T *>(b.p);
    }
    void upload(const std::vector<T> &h, cudaStream_t st) {
        reserve(std::max<size_t>(h.size(), 1), 0, st);
        if (!h.empty()) CK(cudaMemcpyAsync(p, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, st));
    }
};

inline unsigned nblk(uint64_t n, unsigned t) { return (unsigned)((n + t - 1) / t); }

}  // namespace

struct skb_ctx {
    int device = 0;
    cudaStream_t st = nullptr, st_copy = nullptr;
    std::vector<cudaEvent_t> up_ev;
    skb_params prm;
    std::string err;
    int64_t launches = 0;
    int sm_count = 148;
    bool ani_attr_set = false;
    int32_t estimator = SKB_ANI_MEAN;  // skb_set_ani_estimator; kept across skb_clear
    bool ci = false;                   // skb_set_ani_ci; kept across skb_clear
    bool detailed = false;             // skb_set_detailed; kept across skb_clear
    uint64_t marker_c = C_MARKER;      // skb_set_marker_compression / skb_db_load; kept across skb_clear
    int64_t max_results = 0;           // skb_set_max_results (skb_rect's -n; 0: all); kept across skb_clear
    const skb_edge *last_dev_edges = nullptr;  // device copy of the last triangle/rect result (skb_device_edges)
    int64_t last_n_edges = 0;
    bool last_ci = false, last_detailed = false;       // that call ran with --ci / --detailed ...
    const skb_edge_detail *last_dev_detail = nullptr;  // ... and, with either, left the edges' details here
                                                       // (skb_last_edge_ci, skb_last_edge_detail)
    uint64_t genome_set = 0;       // bumped by every call that adds, removes or clears genomes
    int64_t whole_triangle = -1;   // genome_set of the whole skb_triangle that made last_dev_edges, else -1
                                   // (skb_write_matrix with edges == NULL)
    char *h_matrix[2] = {};        // pinned text of two row blocks (skb_write_matrix)
    size_t h_matrix_cap[2] = {};
    std::vector<cudaEvent_t> anchor_ev;  // start/stop pairs around the anchor kernel launches of the current call
    int anchor_ev_used = 0;
    float last_ms_anchor = 0;
    int last_anchor_launches = 0;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    cudaEvent_t call_ev[5] = {};  // start, pairs ready, edges ready of one screen or edge call, and around its -n stage
                                  // (call_events)

    // ---- sketch DB (host metadata; the seeds and raw marker keys themselves are d_seeds, d_mkeys)
    struct SketchDb {
        std::vector<uint64_t> seed_off{0};  // [n+1]
        std::vector<uint64_t> total_len;    // [n]
        std::vector<uint32_t> ctg_off{0};   // [n+1]
        std::vector<uint32_t> ctg_len;      // kept contig lengths
        uint64_t n_mkeys = 0;               // raw marker keys so far

        int32_t n() const { return (int32_t)total_len.size(); }
        template <typename L>
        void append(uint64_t n_seeds, uint64_t len, const L *ctg_lens, size_t n_ctg) {
            seed_off.push_back(seed_off.back() + n_seeds);
            total_len.push_back(len);
            for (size_t k = 0; k < n_ctg; k++) ctg_len.push_back((uint32_t)ctg_lens[k]);
            ctg_off.push_back((uint32_t)ctg_len.size());
        }
        void truncate(int32_t n, uint64_t mkeys) {
            seed_off.resize(n + 1);
            total_len.resize(n);
            ctg_off.resize(n + 1);
            ctg_len.resize(ctg_off.back());
            n_mkeys = mkeys;
        }
        void clear() { *this = SketchDb(); }
    } db;
    // ---- host side of the index skb_index / skb_index_append built over genomes [0, n_indexed)
    struct HostIndex {
        int32_t n_indexed = 0;
        int32_t n_inv_genomes = 0;     // genomes covered by the inverted marker index
        uint64_t n_inv = 0;            // its entries
        uint64_t n_mkeys_indexed = 0;  // raw marker keys consumed by the last (append) index
        std::vector<uint64_t> tab_off{0}, marker_off{0};  // [n_indexed+1]
        std::vector<uint32_t> chunk_off{0};               // [n_indexed+1]
        std::vector<uint32_t> tab_buckets;                // [n_indexed]
        std::vector<uint32_t> ctg_pstart, chunk_start, chunk_len;

        // drop the genomes a truncated sketch DB no longer holds
        void truncate(const SketchDb &db) {
            const int32_t n = db.n();
            if (n_indexed <= n) return;
            n_indexed = n;
            tab_off.resize(n + 1);
            tab_buckets.resize(n);
            ctg_pstart.resize(db.ctg_len.size());
            chunk_off.resize(n + 1);
            chunk_start.resize(chunk_off.back());
            chunk_len.resize(chunk_off.back());
            marker_off.resize(n + 1);
            n_mkeys_indexed = std::min(n_mkeys_indexed, db.n_mkeys);
        }
        void clear() { *this = HostIndex(); }
    } ix;
    // ---- device arrays
    DevBuf<uint64_t> d_seeds, d_mkeys;
    // built by skb_index
    bool indexed = false;
    int32_t own_first = 0, own_count = -1;  // genomes whose seed tables this context builds (skb_set_owned); -1: all
    // seed tables built by skb_index_seed_tables and carried across skb_clear_keep_tables: valid for a context that owns
    // exactly these genomes (count, seed records, table density)
    int32_t kept_n = 0;
    uint64_t kept_seeds = 0;
    int kept_x2 = 0;
    int tab_x2 = 4;        // seed-table buckets per seed, times two: 4 / 2 / 1 = 0.5 / 1 / 2 records per 4-slot bucket
    int tab_x2_forced = 0; // SKB_TAB_X2 (tests exercise the overflow chain with 1)
    int x2_decided = 0;    // density chosen from the free device memory the last time it was asked for ...
    uint64_t x2_decided_seeds = 0;  // ... and the owned seed count it was chosen for
    double x2_budget = 0;           // ... and the table budget in bytes it was chosen under ...
    double x2_room = 0;             // ... and the device memory free for the tables then (table_budget)
    // on-demand seed tables (skb_index chose them: the tables of all genomes exceed the budget): d_tab holds the tables
    // of one block of genomes at a time, built by the edge call that needs them (table_blocks)
    bool on_demand = false;
    int32_t blocks_last_call = 0;   // blocks the last edge call built (skb_table_blocks)
    double block_budget = 0;        // bytes one block may take, once measured after skb_index (block_budget); 0: unknown
    DevBuf<uint64_t> d_seed_off, d_tab, d_tab_off, d_total_len, d_inv, d_markers, d_marker_off;
    DevBuf<uint32_t> d_tab_buckets;
    DevBuf<uint32_t> d_chunk_begin, d_chunk_start, d_chunk_len, d_chunk_off, d_ctg_pstart, d_ctg_len, d_ctg_off,
        d_marker_cnt;
    struct AddCall { int32_t n_before; uint64_t mkeys_before; };
    std::vector<AddCall> add_calls;        // for skb_pop_last_add
    // scratch
    DevBuf<unsigned char> d_tmp;
    std::map<std::string, DevBuf<unsigned char>> pool;  // named scratch, see PoolRef
    DevBuf<int> d_counter;
    DevBuf<PairInfo> d_info;
    DevBuf<uint32_t> d_nch, d_task_off;

    int32_t n() const { return db.n(); }
    bool owns(int32_t g) const { return own_count < 0 || (g >= own_first && g < own_first + own_count); }
    // the owned genomes among [g0, n): one id range [first, second)
    std::pair<int32_t, int32_t> owned_in(int32_t g0, int32_t n) const {
        const int32_t o0 = std::clamp(own_count < 0 ? g0 : own_first, g0, n);
        return {o0, std::clamp(own_count < 0 ? n : own_first + own_count, o0, n)};
    }
    DbView view() const {
        DbView v;
        v.n_genomes = ix.n_indexed;
        v.seeds = d_seeds.p;
        v.g_seed_off = d_seed_off.p;
        v.tab = d_tab.p;
        v.g_tab_off = d_tab_off.p;
        v.g_tab_buckets = d_tab_buckets.p;
        v.chunk_begin = d_chunk_begin.p;
        v.chunk_start = d_chunk_start.p;
        v.chunk_len = d_chunk_len.p;
        v.g_chunk_off = d_chunk_off.p;
        v.ctg_pstart = d_ctg_pstart.p;
        v.ctg_len = d_ctg_len.p;
        v.g_ctg_off = d_ctg_off.p;
        v.g_total_len = d_total_len.p;
        v.markers = d_markers.p;
        v.g_marker_off = d_marker_off.p;
        v.inv_keys = d_inv.p;
        v.n_inv = (int64_t)ix.n_inv;
        return v;
    }
    AniParams ani_params() const {
        AniParams a;
        a.band_bp = prm.band_bp;
        a.max_gap = prm.max_gap;
        a.anchor_score = prm.anchor_score;
        a.min_anchors = prm.min_anchors;
        a.min_score = prm.min_score;
        a.max_mult = prm.max_mult;
        a.max_chunk_chains = prm.max_chunk_chains;
        a.ovl_num = prm.ovl_num;
        a.ovl_den = prm.ovl_den;
        a.span_ext = prm.span_ext;
        a.debias_a = prm.debias_a;
        a.debias_g = prm.debias_g;
        return a;
    }
};

namespace {

template <typename F>
int guarded(skb_ctx *ctx, F &&f) {
    if (!ctx) return SKB_EINVAL;
    try {
        CK(cudaSetDevice(ctx->device));
        return f();
    } catch (const CudaFail &e) {
        ctx->err = e.msg;
        return SKB_ECUDA;
    } catch (const std::bad_alloc &) {
        ctx->err = "host out of memory";
        return SKB_ENOMEM;
    } catch (const std::exception &e) {
        ctx->err = e.what();
        return SKB_EINVAL;
    }
}

int fail(skb_ctx *ctx, int code, const std::string &m) {
    ctx->err = m;
    return code;
}

// Every kernel launch of the library: enqueued on the context's stream and counted (skb_stats.launches).  `kern` may be
// a pointer to one of a kernel's instantiations chosen at run time.
template <typename K, typename... A>
void launch(skb_ctx *c, K kern, dim3 grid, dim3 block, size_t smem, A... args) {
    kern<<<grid, block, smem, c->st>>>(args...);
    CK(cudaGetLastError());
    c->launches++;
}

// A CUB device call f(tmp, bytes): once for the temp size, once on the context's d_tmp.  CUB does not report its
// launches; n_launches is the caller's estimate of them.
template <typename F>
void cub_run(skb_ctx *c, int n_launches, F &&f) {
    size_t bytes = 0;
    CK(f(nullptr, bytes));
    c->d_tmp.reserve(bytes + 16, 0, c->st);
    CK(f(c->d_tmp.p, bytes));
    c->launches += n_launches;
}

void exclusive_scan_u32(skb_ctx *c, const uint32_t *in, uint32_t *out, size_t n) {
    cub_run(c, 2, [&](void *tmp, size_t &bytes) {
        return cub::DeviceScan::ExclusiveSum(tmp, bytes, in, out, (int)n, c->st);
    });
}

__global__ void widen_u8_kernel(const uint8_t *__restrict__ in, uint32_t *__restrict__ out, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i];
}
// out[i] = sum of in[0..i), in place over the widened copy
void exclusive_scan_u8(skb_ctx *c, const uint8_t *in, uint32_t *out, size_t n) {
    launch(c, widen_u8_kernel, (unsigned)((n + 255) / 256), 256, 0, in, out, n);
    exclusive_scan_u32(c, out, out, n);
}

// stable LSD radix sort on key bits [begin_bit, end_bit)
void sort_keys_u64(skb_ctx *c, const uint64_t *in, uint64_t *out, size_t n, int end_bit = 64, int begin_bit = 0) {
    cub_run(c, (end_bit - begin_bit + 7) / 8 + 1, [&](void *tmp, size_t &bytes) {
        return cub::DeviceRadixSort::SortKeys(tmp, bytes, in, out, (int64_t)n, begin_bit, end_bit, c->st);
    });
}

// stable radix sort of (key, value) pairs on key bits [0, end_bit), counted as sort_keys_u64 counts its sort
template <typename K>
void sort_pairs(skb_ctx *c, K *keys_in, K *keys_out, uint32_t *vals_in, uint32_t *vals_out, size_t n,
                int end_bit = 8 * sizeof(K)) {
    cub_run(c, (end_bit + 7) / 8 + 1, [&](void *tmp, size_t &bytes) {
        return cub::DeviceRadixSort::SortPairs(tmp, bytes, keys_in, keys_out, vals_in, vals_out, (int64_t)n, 0, end_bit,
                                               c->st);
    });
}

// kernels cub::DeviceSegmentedSort launches for one call, at most: the partition of the segments by size (two), then the
// large- and the small/medium-segment sorts (a call with few segments runs one kernel instead)
constexpr int EST_SORT_LAUNCHES = 4;

// stable sort of (key, value) pairs within each of the segments [off[s], off[s + 1]), s < n_seg
void segmented_sort_pairs(skb_ctx *c, unsigned long long *keys_in, unsigned long long *keys_out, uint32_t *vals_in,
                          uint32_t *vals_out, int n, int n_seg, uint32_t *off) {
    cub_run(c, EST_SORT_LAUNCHES, [&](void *tmp, size_t &bytes) {
        return cub::DeviceSegmentedSort::StableSortPairs(tmp, bytes, keys_in, keys_out, vals_in, vals_out, n, n_seg, off,
                                                         off + 1, c->st);
    });
}

// ---- sketch a batch of packed genomes [g0, g1) of the caller's list ------------------------------
struct BatchMeta {
    SketchBatch b;
    uint32_t n_tiles = 0;
    size_t n_warps = 0;
    size_t n_ctg = 0;  // contigs of the batch (ctg_start entries)
};

// Host-side layout of a batch -> device, one copy per batch (slot = position in the super-batch).  Issued for every
// batch BEFORE the packed words are enqueued: small copies share the H2D copy engine with the 256 MB word copies,
// and queued behind them they held every sketch kernel back until the last word copy had finished.
BatchMeta sketch_meta(skb_ctx *c, const skb_packed *const *gen, int32_t g0, int32_t g1, const uint64_t *d_words, size_t slot) {
    const int32_t nb = g1 - g0;
    std::vector<uint64_t> word_off(nb + 1, 0), nbases(nb), ctg_start;
    std::vector<uint32_t> ctg_off(nb + 1, 0), tile_off(nb + 1, 0);
    for (int32_t i = 0; i < nb; i++) {
        const skb_packed *p = gen[g0 + i];
        word_off[i + 1] = word_off[i] + (uint64_t)p->n_words;
        nbases[i] = (uint64_t)p->n_bases;
        uint64_t s = 0;
        for (int32_t k = 0; k < p->n_contigs; k++) {
            ctg_start.push_back(s);
            s += (uint64_t)p->contig_lens[k];
        }
        ctg_off[i + 1] = (uint32_t)ctg_start.size();
        tile_off[i + 1] = tile_off[i] + (uint32_t)std::max<uint64_t>(1, (nbases[i] + SK_TILE_BASES - 1) / SK_TILE_BASES);
    }
    // u64 word_off[nb+1] | u64 nbases[nb] | u64 ctg_start[] | u32 ctg_off[nb+1] | u32 tile_off[nb+1]
    const size_t o_nb = (size_t)nb + 1, o_cs = o_nb + (size_t)nb, o_co = o_cs + ctg_start.size();
    const size_t n32 = (size_t)nb + 1, o_to = o_co + (n32 + 1) / 2;
    std::vector<uint64_t> blob(o_to + (n32 + 1) / 2, 0);
    std::copy(word_off.begin(), word_off.end(), blob.begin());
    std::copy(nbases.begin(), nbases.end(), blob.begin() + o_nb);
    std::copy(ctg_start.begin(), ctg_start.end(), blob.begin() + o_cs);
    std::memcpy(blob.data() + o_co, ctg_off.data(), n32 * 4);
    std::memcpy(blob.data() + o_to, tile_off.data(), n32 * 4);
    PoolRef<uint64_t> d_meta(c->pool["sketch_meta." + std::to_string(slot)]);
    d_meta.upload(blob, c->st);
    BatchMeta m;
    m.n_tiles = tile_off[nb];
    m.n_warps = (size_t)m.n_tiles * SK_WARPS;
    m.n_ctg = ctg_start.size();
    m.b.packed = d_words;
    m.b.g_word_off = d_meta.p;
    m.b.g_nbases = d_meta.p + o_nb;
    m.b.ctg_start = d_meta.p + o_cs;
    m.b.g_ctg_off = reinterpret_cast<const uint32_t *>(d_meta.p + o_co);
    m.b.tile_off = reinterpret_cast<const uint32_t *>(d_meta.p + o_to);
    m.b.n = nb;
    m.b.first_gid = 0;  // set when the batch runs
    return m;
}

// per_seq (skb_add_sequences): every contig of the batch is appended as a genome of its own
void sketch_batch(skb_ctx *c, const skb_packed *const *gen, int32_t g0, int32_t g1, const BatchMeta &meta,
                  cudaEvent_t uploaded, bool per_seq) {
    const int32_t nb = g1 - g0;
    const uint32_t n_tiles = meta.n_tiles;
    const size_t n_warps = meta.n_warps;
    PoolRef<uint32_t> d_cnt_s(c->pool["sketch_batch.d_cnt_s"]), d_cnt_m(c->pool["sketch_batch.d_cnt_m"]), d_off_s(c->pool["sketch_batch.d_off_s"]), d_off_m(c->pool["sketch_batch.d_off_m"]);
    CK(cudaStreamWaitEvent(c->st, uploaded, 0));  // the batch's words were enqueued on the copy stream
    d_cnt_s.reserve(n_warps + 1, 0, c->st);
    d_cnt_m.reserve(n_warps + 1, 0, c->st);
    d_off_s.reserve(n_warps + 1, 0, c->st);
    d_off_m.reserve(n_warps + 1, 0, c->st);
    CK(cudaMemsetAsync(d_cnt_s.p + n_warps, 0, 4, c->st));
    CK(cudaMemsetAsync(d_cnt_m.p + n_warps, 0, 4, c->st));
    SketchBatch b = meta.b;
    b.first_gid = (uint32_t)c->n();
    b.thr_marker = marker_threshold(c->marker_c);
    PoolRef<ulonglong2> d_masks(c->pool["sketch_batch.d_masks"]);
    d_masks.reserve(n_warps * 32, 0, c->st);
    launch(c, sketch_kernel<false>, n_tiles, SK_THREADS, 0, b, d_cnt_s.p, d_cnt_m.p, nullptr, nullptr, nullptr, nullptr,
           d_masks.p);
    exclusive_scan_u32(c, d_cnt_s.p, d_off_s.p, n_warps + 1);
    exclusive_scan_u32(c, d_cnt_m.p, d_off_m.p, n_warps + 1);
    // per-genome seed offsets = scanned offsets at genome tile boundaries; per-sequence: at every contig's first base
    const size_t n_units = per_seq ? meta.n_ctg : (size_t)nb;
    std::vector<uint32_t> h_off_s(n_units + 1);
    uint32_t tot_m = 0;
    PoolRef<uint32_t> d_goff(c->pool["sketch_batch.d_goff"]);
    d_goff.reserve(n_units + 1, 0, c->st);
    if (per_seq)
        launch(c, record_seed_off_kernel, nblk((uint64_t)n_units + 1, 256), 256, 0, b, d_off_s.p, d_masks.p,
               (int)n_units, n_warps, d_goff.p);
    else
        launch(c, gather_strided_kernel, nblk((uint64_t)nb + 1, 256), 256, 0, d_off_s.p, b.tile_off, SK_WARPS, nb + 1,
               d_goff.p);
    CK(cudaMemcpyAsync(h_off_s.data(), d_goff.p, (n_units + 1) * 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaMemcpyAsync(&tot_m, d_off_m.p + n_warps, 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    const uint64_t cur_seeds = c->db.seed_off.back();
    const uint64_t tot_s = h_off_s[n_units];
    c->d_seeds.reserve(cur_seeds + tot_s + 1, cur_seeds, c->st);
    c->d_mkeys.reserve(c->db.n_mkeys + tot_m + 1, c->db.n_mkeys, c->st);
    launch(c, per_seq ? sketch_kernel<true, true> : sketch_kernel<true>, n_tiles, SK_THREADS, 0, b, nullptr, nullptr,
           d_off_s.p, d_off_m.p, c->d_seeds.p + cur_seeds, c->d_mkeys.p + c->db.n_mkeys, d_masks.p);
    CK(cudaStreamSynchronize(c->st));  // batch-local buffers die here
    size_t u = 0;
    for (int32_t i = 0; i < nb; i++) {
        const skb_packed *p = gen[g0 + i];
        if (!per_seq) {
            c->db.append(h_off_s[u + 1] - h_off_s[u], (uint64_t)p->n_bases, p->contig_lens, (size_t)p->n_contigs);
            u++;
        } else
            for (int32_t k = 0; k < p->n_contigs; k++, u++)
                c->db.append(h_off_s[u + 1] - h_off_s[u], (uint64_t)p->contig_lens[k], p->contig_lens + k, 1);
    }
    c->db.n_mkeys += tot_m;
    c->indexed = false;
}

// ---- ANI over a device-resident pair list --------------------------------------------------------
// Scratch of the pair stage, kept across calls (no cudaMalloc/cudaFree in the steady state).
//   info      : roles and chunk count per pair
//   task_off  : exclusive prefix of chunk counts -> task id = (pair, chunk)
//   cands     : SLOTS candidate slots per task;  task_ncand: how many are filled

// d_ci: nullptr, or [n_pairs] for every pair's --ci interval (ci_kernel), indexed like d_out
// d_sd: nullptr, or (with d_ci) [n_pairs] for every pair's --detailed standard deviation (sd_kernel), indexed like d_out
void run_ani(skb_ctx *c, const unsigned long long *d_pairs, int64_t n_pairs, PairOut *d_out, double2 *d_ci = nullptr,
             double *d_sd = nullptr) {
    c->anchor_ev_used = 0;
    if (n_pairs == 0) return;
    if (n_pairs >= (1ll << 31)) throw CudaFail{"too many surviving pairs in one call"};
    // candidates per pair the warp-per-pair finalize kernel keeps in shared memory (a multiple of 32)
    static const uint32_t fw_cap = [] {
        const char *e = std::getenv("SKB_FW_CAP");
        const int v = e ? atoi(e) : 1024;
        uint32_t w = 32;
        while ((int)w < v && w < 4096) w <<= 1;  // a power of two: the bitonic network's size
        return w;
    }();
    const size_t fw_smem = (size_t)FW_WARPS * ((fw_bytes_per_warp(fw_cap) + 15) & ~(size_t)15);
    if (!c->ani_attr_set) {
        CK(cudaFuncSetAttribute(finalize_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)(FIN_BYTES_PER_CAND * MAXP)));
        CK(cudaFuncSetAttribute(finalize_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)(FIN_BYTES_PER_CAND * MAXP)));
        CK(cudaFuncSetAttribute(finalize_warp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fw_smem));
        CK(cudaFuncSetAttribute(finalize_warp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fw_smem));
        c->ani_attr_set = true;
    }
    // median / robust: the finalize kernels also store every candidate's accepted flag, and an estimator stage per
    // batch turns the accepted chains into one ANI (est_key_kernel, segmented sort, est_pick_kernel)
    const bool est = c->estimator != SKB_ANI_MEAN;
    // --ci (and --detailed, which prints the interval too): the accepted flags too, and ci_kernel per batch bootstraps
    // the pair's accepted chains; --detailed's sd_kernel then reads the chain list ci_kernel compacted
    const bool acc = est || d_ci;
    const DbView view = c->view();
    const AniParams prm = c->ani_params();
    c->d_info.reserve((size_t)n_pairs, 0, c->st);
    c->d_nch.reserve((size_t)n_pairs + 1, 0, c->st);
    c->d_task_off.reserve((size_t)n_pairs + 1, 0, c->st);
    PoolRef<unsigned long long> d_key(c->pool["run_ani.key"]), d_key2(c->pool["run_ani.key2"]);
    PoolRef<uint32_t> d_idx(c->pool["run_ani.idx"]), d_perm(c->pool["run_ani.perm"]);
    PoolRef<PairInfo> d_info_s(c->pool["run_ani.info_sorted"]);
    d_key.reserve((size_t)n_pairs, 0, c->st);
    d_key2.reserve((size_t)n_pairs, 0, c->st);
    d_idx.reserve((size_t)n_pairs, 0, c->st);
    d_perm.reserve((size_t)n_pairs, 0, c->st);
    d_info_s.reserve((size_t)n_pairs, 0, c->st);
    launch(c, pair_setup_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, view, d_pairs, n_pairs, c->d_info.p, d_key.p,
           d_idx.p);
    sort_pairs(c, d_key.p, d_key2.p, d_idx.p, d_perm.p, (size_t)n_pairs);
    launch(c, pair_gather_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, c->d_info.p, d_perm.p, n_pairs, d_info_s.p,
           c->d_nch.p);
    // global task offsets (exclusive scan of the chunk counts in processing order)
    CK(cudaMemsetAsync(c->d_nch.p + n_pairs, 0, 4, c->st));
    exclusive_scan_u32(c, c->d_nch.p, c->d_task_off.p, (size_t)n_pairs + 1);
    std::vector<uint32_t> h_nch((size_t)n_pairs);
    CK(cudaMemcpyAsync(h_nch.data(), c->d_nch.p, (size_t)n_pairs * 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    uint64_t total_tasks = 0;
    for (uint32_t v : h_nch) total_tasks += v;
    // task_off is a 32-bit scan and may wrap when a call holds more than 2^32 (pair, chunk) tasks (a single-species set
    // of ~6,000 genomes): every kernel uses task_off[p] - base within one batch of <= 8 Mi tasks, which is exact
    // modulo 2^32.
    // Batches of pairs bound the scratch (<= 8 Mi tasks per batch) and keep a batch's reference tables and
    // candidates warm in L2 between its kernels.  One in-order stream: running the anchor kernel of batch b+1 beside
    // chain/finalize of batch b on a second stream was measured slower in every configuration (round 1, DESIGN.md).
    // About 5 Mi tasks per batch (SKB_PAIR_BATCH_TASKS): six batches for config3 on one GPU (measured best there), one
    // for an eighth of it -- every batch costs ~0.3 ms of launches, scans and one host round trip.
    static const uint64_t batch_tasks = [] {
        const char *e = std::getenv("SKB_PAIR_BATCH_TASKS");
        return (uint64_t)(e ? std::max(1 << 16, atoi(e)) : (5 << 20));
    }();
    const uint64_t want_batches = std::max<uint64_t>(1, (total_tasks + batch_tasks / 2) / batch_tasks);
    const uint64_t max_tasks = std::min<uint64_t>(8ull << 20, (total_tasks + want_batches - 1) / want_batches + 4096);
    struct Batch { int64_t p0, p1; uint64_t base, tasks; };
    std::vector<Batch> batches;
    {
        int64_t p0 = 0;
        uint64_t base = 0;
        while (p0 < n_pairs) {
            uint64_t tasks = 0;
            int64_t p1 = p0;
            while (p1 < n_pairs && (p1 == p0 || tasks + h_nch[(size_t)p1] <= max_tasks)) tasks += h_nch[(size_t)p1++];
            if (tasks >= (1ull << 32)) throw CudaFail{"one pair has more than 2^32 query chunks"};
            batches.push_back({p0, p1, base, tasks});
            base += tasks;
            p0 = p1;
        }
    }
    uint64_t cap = 1;
    int64_t cap_pairs = 1;
    for (const Batch &bt : batches) {
        cap = std::max(cap, bt.tasks);
        cap_pairs = std::max(cap_pairs, bt.p1 - bt.p0);
    }
    PoolRef<uint64_t> b_anc(c->pool["ani.anc"]);
    PoolRef<uint32_t> b_res(c->pool["ani.res"]), b_next(c->pool["ani.next"]), b_fctl(c->pool["ani.fin_ctl"]),
        b_big_list(c->pool["ani.big_list"]), b_big_nc(c->pool["ani.big_nc"]), b_mid_list(c->pool["ani.mid_list"]);
    PoolRef<uint16_t> b_tn(c->pool["ani.tn"]);
    PoolRef<TaskDesc> b_desc(c->pool["ani.desc"]);
    PoolRef<Cand> b_cands(c->pool["ani.cands"]);
    PoolRef<PCand> b_pcands(c->pool["ani.pcands"]);
    PoolRef<uint32_t> b_task_pair(c->pool["ani.task_pair"]), b_cand_off(c->pool["ani.cand_off"]);
    PoolRef<uint8_t> b_ncand(c->pool["ani.ncand"]);
    PoolRef<uint32_t> b_slow(c->pool["ani.slow_list"]);
    b_anc.reserve(slab_entries(cap) + 2, 0, c->st);
    b_res.reserve(slab_entries(cap), 0, c->st);
    b_tn.reserve((size_t)cap, 0, c->st);
    b_desc.reserve((size_t)cap, 0, c->st);
    b_cands.reserve((size_t)cap * SLOTS, 0, c->st);
    b_pcands.reserve((size_t)cap * SLOTS, 0, c->st);
    b_task_pair.reserve((size_t)cap, 0, c->st);
    b_cand_off.reserve((size_t)cap + 1, 0, c->st);
    b_ncand.reserve((size_t)cap + 1, 0, c->st);
    b_slow.reserve((size_t)cap + 1, 0, c->st);
    b_next.reserve(1, 0, c->st);
    b_fctl.reserve(4, 0, c->st);
    b_mid_list.reserve((size_t)cap_pairs, 0, c->st);
    b_big_list.reserve((size_t)cap_pairs, 0, c->st);
    b_big_nc.reserve((size_t)cap_pairs, 0, c->st);
    PoolRef<uint8_t> e_acc(c->pool["est.acc"]);
    if (acc) e_acc.reserve((size_t)cap * SLOTS, 0, c->st);
    // When no padded position of the database comes near 2^30, anchor_kernel matches and decodes seed records by their
    // 32-bit halves and chain_kernel compares diagonals (reference position -/+ query position, sign by strand) in 32
    // bits; SKB_WIDE_DIAG=1 forces the general variants (tests run both)
    bool wide_diag = std::getenv("SKB_WIDE_DIAG") != nullptr && atoi(std::getenv("SKB_WIDE_DIAG")) != 0;
    for (int32_t g = 0; g < c->ix.n_indexed && !wide_diag; g++) {
        const uint32_t k1 = c->db.ctg_off[(size_t)g + 1];
        if (k1 > c->db.ctg_off[(size_t)g] &&
            (uint64_t)c->ix.ctg_pstart[k1 - 1] + c->db.ctg_len[k1 - 1] >= (1ull << 30) - (1ull << 21))
            wide_diag = true;
    }
    static const bool trace = std::getenv("SKB_TRACE") != nullptr;  // diagnosis: per-kernel timeline on stderr
    struct Span { const char *name; size_t batch; cudaEvent_t e0, e1; };
    std::vector<Span> spans;
    cudaEvent_t ev_t0 = nullptr;
    auto mark = [&]() {
        cudaEvent_t e = nullptr;
        if (trace) {
            CK(cudaEventCreate(&e));
            CK(cudaEventRecord(e, c->st));
        }
        return e;
    };
    if (trace) ev_t0 = mark();
    for (size_t bi = 0; bi < batches.size(); bi++) {
        const Batch &bt = batches[bi];
        const int64_t np = bt.p1 - bt.p0;
        const uint32_t tasks = (uint32_t)bt.tasks, base = (uint32_t)bt.base;
        CK(cudaMemsetAsync(b_fctl.p, 0, 16, c->st));
        if (tasks) {
            CK(cudaMemsetAsync(b_ncand.p, 0, (size_t)tasks + 1, c->st));
            CK(cudaMemsetAsync(b_slow.p, 0, 4, c->st));
            CK(cudaMemsetAsync(b_next.p, 0, 4, c->st));
            launch(c, task_setup_kernel, nblk(tasks, 256), 256, 0, view, d_info_s.p + bt.p0, c->d_task_off.p + bt.p0, base, np,
                   tasks, b_desc.p, b_task_pair.p);
            // a persistent grid fed by the task counter
            const unsigned g1 = std::min<unsigned>(nblk(tasks, (ANC_THREADS / 32) * ANC_GRAB), (unsigned)c->sm_count * 32u);
            if ((int)c->anchor_ev.size() < c->anchor_ev_used + 2) {
                cudaEvent_t e0, e1;
                CK(cudaEventCreate(&e0));
                CK(cudaEventCreate(&e1));
                c->anchor_ev.push_back(e0);
                c->anchor_ev.push_back(e1);
            }
            CK(cudaEventRecord(c->anchor_ev[c->anchor_ev_used], c->st));
            cudaEvent_t t0 = mark();
            launch(c, wide_diag ? anchor_kernel<false> : anchor_kernel<true>, g1, ANC_THREADS, 0, view, prm, b_desc.p, tasks,
                   b_anc.p, b_tn.p, b_next.p);
            if (trace) spans.push_back({"anchor", bi, t0, mark()});
            CK(cudaEventRecord(c->anchor_ev[c->anchor_ev_used + 1], c->st));
            c->anchor_ev_used += 2;
            t0 = mark();
            launch(c, wide_diag ? chain_kernel<true> : chain_kernel<false>, nblk(tasks, DP_THREADS), DP_THREADS, 0, prm, tasks,
                   b_anc.p, b_tn.p, b_res.p, b_desc.p, b_cands.p, b_ncand.p, b_slow.p);
            if (trace) spans.push_back({"chain", bi, t0, mark()});
            const unsigned g3 = std::min<unsigned>(nblk(tasks, END_THREADS / 32), (unsigned)c->sm_count * 4u);
            launch(c, ends_kernel, g3, END_THREADS, 0, prm, tasks, b_anc.p, b_res.p, b_tn.p, b_desc.p, b_slow.p, b_cands.p,
                   b_ncand.p);
        }
        cudaEvent_t tf = mark();
        // selection + ANI/AF: a warp per pair; the kernel lists the pairs it leaves to the CTA-per-pair kernels
        if (tasks) {
            exclusive_scan_u8(c, b_ncand.p, b_cand_off.p, (size_t)tasks + 1);  // b_ncand[tasks] = 0
            launch(c, cand_pack_kernel, nblk(tasks, 256), 256, 0, view, prm, d_info_s.p + bt.p0, tasks, b_task_pair.p, b_ncand.p,
                   b_cand_off.p, b_cands.p, b_pcands.p);
        }
        launch(c, acc ? finalize_warp_kernel<true> : finalize_warp_kernel<false>, nblk((uint64_t)np, FW_WARPS), FW_WARPS * 32,
               fw_smem, view, prm, d_info_s.p + bt.p0, c->d_task_off.p + bt.p0, base, np, b_pcands.p, b_cand_off.p,
               d_perm.p + bt.p0, d_out, fw_cap, b_fctl.p, b_mid_list.p, b_big_list.p, b_big_nc.p, e_acc.p);
        uint32_t fctl[4] = {0, 0, 0, 0};
        uint32_t n_cand = 0;
        CK(cudaMemcpyAsync(fctl, b_fctl.p, 16, cudaMemcpyDeviceToHost, c->st));
        if (est && tasks) CK(cudaMemcpyAsync(&n_cand, b_cand_off.p + tasks, 4, cudaMemcpyDeviceToHost, c->st));
        CK(cudaStreamSynchronize(c->st));
        if (fctl[2]) {  // more than fw_cap candidates or more than FW_EDGES blocking relations: shared memory, one CTA per pair
            uint32_t fcap = 32;
            while (fcap < fctl[0]) fcap <<= 1;
            launch(c, acc ? finalize_kernel<false, true> : finalize_kernel<false, false>, fctl[2], FIN_THREADS,
                   FIN_BYTES_PER_CAND * (size_t)fcap, view, prm, d_info_s.p + bt.p0, c->d_task_off.p + bt.p0, base, np,
                   b_pcands.p, b_cand_off.p, d_perm.p + bt.p0, d_out, fcap, b_mid_list.p, nullptr, nullptr, nullptr, e_acc.p);
        }
        if (fctl[1]) {  // pairs beyond MAXP candidates: same kernel body on global scratch, one CTA per pair
            const uint32_t nbig = fctl[1];
            std::vector<uint32_t> h_nc(nbig), h_cap(nbig);
            std::vector<unsigned long long> h_off(nbig);
            CK(cudaMemcpyAsync(h_nc.data(), b_big_nc.p, (size_t)nbig * 4, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            unsigned long long off = 0;
            for (uint32_t k = 0; k < nbig; k++) {
                uint32_t m = 32;
                while (m < h_nc[k]) m <<= 1;
                if (m > FIN_IDX_MASK) throw CudaFail{"a pair has more than 2^24 chain candidates"};
                h_cap[k] = m;
                h_off[k] = off;
                off += (unsigned long long)FIN_BYTES_PER_CAND * m;
                off = (off + 255) & ~255ull;
            }
            PoolRef<unsigned char> d_big(c->pool["ani.big_scratch"]);
            PoolRef<unsigned long long> d_big_off(c->pool["ani.big_off"]);
            PoolRef<uint32_t> d_big_cap(c->pool["ani.big_cap"]);
            d_big.reserve((size_t)off + 256, 0, c->st);
            d_big_off.upload(h_off, c->st);
            d_big_cap.upload(h_cap, c->st);
            launch(c, acc ? finalize_kernel<true, true> : finalize_kernel<true, false>, nbig, FIN_THREADS, 0, view, prm,
                   d_info_s.p + bt.p0, c->d_task_off.p + bt.p0, base, np, b_pcands.p, b_cand_off.p, d_perm.p + bt.p0, d_out, 0,
                   b_big_list.p, d_big_off.p, d_big_cap.p, d_big.p, e_acc.p);
            CK(cudaStreamSynchronize(c->st));  // h_off / h_cap leave scope
        }
        if (trace) spans.push_back({"finalize", bi, tf, mark()});
        if (d_ci) {
            cudaEvent_t tc = mark();
            PoolRef<uint32_t> ci_chains(c->pool["ci.chains"]);
            ci_chains.reserve((size_t)cap * SLOTS, 0, c->st);
            launch(c, ci_kernel, nblk((uint64_t)np, FW_WARPS), FW_WARPS * 32, 0, prm, d_info_s.p + bt.p0,
                   c->d_task_off.p + bt.p0, base, np, b_pcands.p, b_cand_off.p, e_acc.p, ci_chains.p, d_perm.p + bt.p0, d_out,
                   d_ci);
            if (trace) spans.push_back({"ci", bi, tc, mark()});
            if (d_sd) {
                cudaEvent_t ts = mark();
                launch(c, sd_kernel, nblk((uint64_t)np, FW_WARPS), FW_WARPS * 32, 0, prm, c->d_task_off.p + bt.p0, base, np,
                       b_cand_off.p, ci_chains.p, d_perm.p + bt.p0, d_out, d_sd);
                if (trace) spans.push_back({"detail", bi, ts, mark()});
            }
        }
        if (est && n_cand) {
            cudaEvent_t te = mark();
            PoolRef<unsigned long long> e_key(c->pool["est.key"]), e_key_s(c->pool["est.key_sorted"]);
            PoolRef<uint32_t> e_idx(c->pool["est.idx"]), e_idx_s(c->pool["est.idx_sorted"]), e_seg(c->pool["est.seg"]);
            e_key.reserve(n_cand, 0, c->st);
            e_key_s.reserve(n_cand, 0, c->st);
            e_idx.reserve(n_cand, 0, c->st);
            e_idx_s.reserve(n_cand, 0, c->st);
            e_seg.reserve((size_t)np + 1, 0, c->st);
            launch(c, est_key_kernel, nblk(std::max<uint64_t>(n_cand, (uint64_t)np + 1), 256), 256, 0, b_pcands.p, e_acc.p,
                   n_cand, c->d_task_off.p + bt.p0, base, np, b_cand_off.p, e_key.p, e_idx.p, e_seg.p);
            segmented_sort_pairs(c, e_key.p, e_key_s.p, e_idx.p, e_idx_s.p, (int)n_cand, (int)np, e_seg.p);
            launch(c, est_pick_kernel, nblk((uint64_t)np, FW_WARPS), FW_WARPS * 32, 0, prm, c->estimator, np, e_seg.p,
                   e_idx_s.p, b_pcands.p, d_perm.p + bt.p0, d_out);
            if (trace) spans.push_back({"estimator", bi, te, mark()});
        }
    }
    if (trace) {
        CK(cudaStreamSynchronize(c->st));
        for (const Span &sp : spans) {
            float a = 0, b = 0;
            CK(cudaEventElapsedTime(&a, ev_t0, sp.e0));
            CK(cudaEventElapsedTime(&b, ev_t0, sp.e1));
            fprintf(stderr, "[skb trace] batch %zu %-8s %8.2f -> %8.2f ms (%.2f)\n", sp.batch, sp.name, a, b, b - a);
            cudaEventDestroy(sp.e0);
            cudaEventDestroy(sp.e1);
        }
        cudaEventDestroy(ev_t0);
    }
}

// pairs on device -> ANI -> compacted edges on device (c->last_dev_edges, c->last_n_edges); sums: sum query seeds, sum
// anchors.  pair_pos, edge_pos (on-demand tables: pairs_to_edges_blocks): a number per pair, copied for every edge
void pairs_to_edges(skb_ctx *c, unsigned long long *d_pairs, int64_t n_pairs, double min_af_pct,
                    unsigned long long sums[2], cudaEvent_t ev_mid, cudaEvent_t ev_end, const uint32_t *pair_pos = nullptr,
                    uint32_t *edge_pos = nullptr) {
    PoolRef<PairOut> d_out(c->pool["pairs_to_edges.d_out"]);
    PoolRef<skb_edge> d_edges(c->pool["pairs_to_edges.d_edges"]);
    PoolRef<unsigned long long> d_n(c->pool["pairs_to_edges.d_n"]);
    d_n.reserve(4, 0, c->st);
    CK(cudaMemsetAsync(d_n.p, 0, 32, c->st));
    CK(cudaEventRecord(ev_mid, c->st));
    c->last_ci = c->ci;
    c->last_detailed = c->detailed;
    c->last_dev_detail = nullptr;
    if (n_pairs > 0) {
        d_out.reserve((size_t)n_pairs, 0, c->st);
        d_edges.reserve((size_t)n_pairs, 0, c->st);
        double2 *d_ci = nullptr;
        if (c->ci || c->detailed) {
            PoolRef<double2> ci_pairs(c->pool["ci.pairs"]);
            ci_pairs.reserve((size_t)n_pairs, 0, c->st);
            d_ci = ci_pairs.p;
        }
        double *d_sd = nullptr;
        if (c->detailed) {
            PoolRef<double> sd_pairs(c->pool["detail.sd"]);
            sd_pairs.reserve((size_t)n_pairs, 0, c->st);
            d_sd = sd_pairs.p;
        }
        run_ani(c, d_pairs, n_pairs, d_out.p, d_ci, d_sd);
        PoolRef<uint32_t> d_ef(c->pool["pairs_to_edges.flag"]), d_ep(c->pool["pairs_to_edges.pos"]);
        d_ef.reserve((size_t)n_pairs, 0, c->st);
        d_ep.reserve((size_t)n_pairs, 0, c->st);
        launch(c, edge_flag_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, d_out.p, n_pairs, min_af_pct / 100.0, d_ef.p);
        exclusive_scan_u32(c, d_ef.p, d_ep.p, (size_t)n_pairs);
        launch(c, edge_scatter_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, d_pairs, d_out.p, n_pairs, d_ef.p, d_ep.p,
               d_edges.p, d_n.p);
        if (edge_pos)
            launch(c, edge_pos_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, d_ef.p, d_ep.p, n_pairs, pair_pos, edge_pos);
        if (d_ci) {  // one record per edge serves both skb_last_edge_ci and skb_last_edge_detail
            PoolRef<skb_edge_detail> det_edges(c->pool["detail.edges"]);
            det_edges.reserve((size_t)n_pairs, 0, c->st);
            launch(c, edge_detail_scatter_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, d_out.p, d_ci, d_sd, n_pairs, d_ef.p,
                   d_ep.p, det_edges.p);
            c->last_dev_detail = det_edges.p;
        }
    }
    CK(cudaEventRecord(ev_end, c->st));
    if (n_pairs > 0)
        launch(c, pair_sums_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, c->d_info.p, d_out.p, n_pairs, c->d_seed_off.p,
               d_n.p + 1);
    unsigned long long h3[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(h3, d_n.p, 32, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    sums[0] = h3[1];
    sums[1] = h3[2];
    c->last_ms_anchor = 0;
    c->last_anchor_launches = c->anchor_ev_used / 2;
    for (int i = 0; i + 1 < c->anchor_ev_used; i += 2) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, c->anchor_ev[i], c->anchor_ev[i + 1]));
        c->last_ms_anchor += ms;
    }
    c->anchor_ev_used = 0;
    c->last_dev_edges = d_edges.p;
    c->last_n_edges = (int64_t)h3[0];
}

// skani's -n (skb_set_max_results): cut the last edge call's list, and its --ci / --detailed records, to each query's
// first max_n edges in row order (query, ANI descending, reference ascending); skb_best_n.cuh.  The kept edges keep
// their (a, b) order.
void best_n_edges(skb_ctx *c, int64_t max_n) {
    const int64_t n = c->last_n_edges;
    PoolRef<unsigned long long> d_key(c->pool["best_n.key"]), d_key_s(c->pool["best_n.key_sorted"]);
    PoolRef<uint32_t> d_idx(c->pool["best_n.idx"]), d_idx_a(c->pool["best_n.idx_ani"]), d_idx_q(c->pool["best_n.idx_row"]);
    PoolRef<uint32_t> d_q(c->pool["best_n.query"]), d_q_s(c->pool["best_n.query_sorted"]);
    PoolRef<uint32_t> d_f(c->pool["best_n.flag"]), d_p(c->pool["best_n.pos"]);
    for (auto *b : {&d_idx, &d_idx_a, &d_idx_q, &d_q, &d_q_s}) b->reserve((size_t)n, 0, c->st);
    d_key.reserve((size_t)n, 0, c->st);
    d_key_s.reserve((size_t)n, 0, c->st);
    d_f.reserve((size_t)n + 1, 0, c->st);
    d_p.reserve((size_t)n + 1, 0, c->st);
    const unsigned nb = nblk((uint64_t)n, 256);
    launch(c, best_n_key_kernel, nb, 256, 0, c->last_dev_edges, n, d_key.p, d_idx.p);
    sort_pairs(c, d_key.p, d_key_s.p, d_idx.p, d_idx_a.p, (size_t)n);
    launch(c, best_n_query_kernel, nb, 256, 0, c->last_dev_edges, d_idx_a.p, n, d_q.p);
    int q_bits = 1;  // query ids are genome ids < n()
    while (q_bits < 32 && (1ll << q_bits) < (int64_t)c->n()) q_bits++;
    sort_pairs(c, d_q.p, d_q_s.p, d_idx_a.p, d_idx_q.p, (size_t)n, q_bits);
    launch(c, best_n_flag_kernel, nb, 256, 0, d_q_s.p, d_idx_q.p, n, max_n, d_f.p);
    CK(cudaMemsetAsync(d_f.p + n, 0, 4, c->st));
    exclusive_scan_u32(c, d_f.p, d_p.p, (size_t)n + 1);
    PoolRef<skb_edge> kept(c->pool["best_n.edges"]);
    kept.reserve((size_t)n, 0, c->st);
    launch(c, best_n_scatter_kernel<skb_edge>, nb, 256, 0, c->last_dev_edges, n, d_f.p, d_p.p, kept.p);
    c->last_dev_edges = kept.p;
    if (c->last_dev_detail) {
        PoolRef<skb_edge_detail> kept_det(c->pool["best_n.detail"]);
        kept_det.reserve((size_t)n, 0, c->st);
        launch(c, best_n_scatter_kernel<skb_edge_detail>, nb, 256, 0, c->last_dev_detail, n, d_f.p, d_p.p, kept_det.p);
        c->last_dev_detail = kept_det.p;
    }
    uint32_t n_kept = 0;
    CK(cudaMemcpyAsync(&n_kept, d_p.p + n, 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    c->last_n_edges = n_kept;
}

// ---- on-demand seed tables (skb_index chose them; DESIGN.md section 2) ------------------------------------------
// Bytes the seed tables may take: table_density's budget, but at least half of the device memory free when it was set
// (a device whose other tenants leave less than the 40 GiB table_density keeps for the rest still holds a small set's
// tables resident), capped by SKB_TABLE_BUDGET_MB (MiB, fractions allowed; tests and benchmarks force on-demand tables
// at small sizes with it)
double table_budget(const skb_ctx *c) {
    const double dev = std::max(c->x2_budget, c->x2_room / 2.0);
    const char *e = std::getenv("SKB_TABLE_BUDGET_MB");
    const double mb = e ? std::strtod(e, nullptr) : 0.0;
    return mb > 0.0 ? std::min(dev, mb * (double)(1ull << 20)) : dev;
}

// Bytes one block of on-demand tables may take: the table budget, and the device memory free now (the scratch allocated
// since the budget was set, such as skb_index's marker sort, is no longer free) less the 40 GiB table_density keeps for
// the pair stage, but at least a tenth of it.  Measured once and kept until skb_index or skb_clear resets it:
// cudaMemGetInfo stalls while a monitoring tool holds the driver lock (table_density), and a search serves many queries.
double block_budget(skb_ctx *c) {
    if (c->block_budget <= 0.0) {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const double room = (double)free_b + (double)c->d_tab.cap * 8.0;
        c->block_budget = std::min(table_budget(c), std::max(room - 40.0 * (double)(1ull << 30), room / 10.0));
    }
    return c->block_budget;
}

// Buckets of genome g's seed table at density tab_x2
uint32_t table_buckets(const skb_ctx *c, int32_t g) {
    const uint64_t ns = c->db.seed_off[g + 1] - c->db.seed_off[g];
    return (uint32_t)std::max<uint64_t>(2, ns * (uint64_t)c->tab_x2 / 2 + 1);
}

// The genomes `ids` (ascending) packed in order into blocks under block_budget; a genome whose table alone exceeds it
// gets a block of its own
std::vector<std::vector<int32_t>> table_blocks(skb_ctx *c, const std::vector<int32_t> &ids) {
    const double budget = block_budget(c);
    std::vector<std::vector<int32_t>> blocks;
    double bytes = 0;
    for (const int32_t g : ids) {
        const double b = (double)c->ix.tab_buckets[g] * BUCKET * 8.0;
        if (blocks.empty() || bytes + b > budget) {
            blocks.emplace_back();
            bytes = 0;
        }
        blocks.back().push_back(g);
        bytes += b;
    }
    return blocks;
}

// The seed tables and repeat flags of one block of genomes (ids ascending), laid out from slot 0 of d_tab; the per-genome
// table offsets and bucket counts of the block's genomes point there (those of the other genomes are stale)
void build_block_tables(skb_ctx *c, const std::vector<int32_t> &ids) {
    const int k = (int)ids.size();
    std::vector<uint32_t> gid(k), nb(k);
    std::vector<uint64_t> loc(k), pref(k + 1, 0);
    uint64_t words = 0;
    for (int j = 0; j < k; j++) {
        const int32_t g = ids[j];
        gid[j] = (uint32_t)g;
        nb[j] = c->ix.tab_buckets[g];
        loc[j] = words;
        words += (uint64_t)nb[j] * BUCKET;
        pref[j + 1] = pref[j] + (c->db.seed_off[g + 1] - c->db.seed_off[g]);
    }
    PoolRef<uint32_t> d_gid(c->pool["table_blocks.gid"]), d_nb(c->pool["table_blocks.nb"]);
    PoolRef<uint64_t> d_loc(c->pool["table_blocks.loc"]), d_pref(c->pool["table_blocks.pref"]);
    d_gid.upload(gid, c->st);
    d_nb.upload(nb, c->st);
    d_loc.upload(loc, c->st);
    d_pref.upload(pref, c->st);
    launch(c, block_layout_kernel, nblk((uint64_t)k, 256), 256, 0, d_gid.p, d_loc.p, d_nb.p, k, c->d_tab_off.p,
           c->d_tab_buckets.p);
    if (words + BUCKET > c->d_tab.cap) {  // the previous block's tables are not needed: free them before growing
        CK(cudaStreamSynchronize(c->st));
        c->d_tab.release();
    }
    c->d_tab.reserve(words + BUCKET, 0, c->st);
    CK(cudaMemsetAsync(c->d_tab.p, 0xFF, words * 8, c->st));
    if (pref[k]) {
        launch(c, block_tab_insert_kernel, nblk(pref[k], 256), 256, 0, c->d_seeds.p, c->d_seed_off.p, d_gid.p, d_pref.p, k,
               c->d_tab.p, c->d_tab_off.p, c->d_tab_buckets.p);
        launch(c, block_rep_flag_kernel, nblk(pref[k], 256), 256, 0, c->d_seeds.p, c->d_seed_off.p, d_gid.p, d_pref.p, k,
               c->d_tab.p, c->d_tab_off.p, c->d_tab_buckets.p, c->prm.max_mult);
    }
}

// The context's events around the stages of one screen or edge call: start, pairs ready, edges ready
cudaEvent_t *call_events(skb_ctx *c) {
    for (cudaEvent_t &e : c->call_ev)
        if (!e) CK(cudaEventCreate(&e));
    return c->call_ev;
}

// The pairs an edge call evaluates (sorted, on the device) and the pair count its stats report as n_pairs_total
struct EdgePairs {
    unsigned long long *d_pairs = nullptr;
    int64_t n = 0, total = 0;
};

// pairs_to_edges with on-demand seed tables: the genomes that are the reference of a pair (ref_mark_kernel) are packed
// into blocks under the table budget; per block its tables are built, its pairs selected in order
// (pair_owned_flag_kernel over the block's id range, which holds no other reference) and evaluated, and its edges (and
// --ci / --detailed records) appended with each edge's position in the pair list; the blocks' lists are then merged by
// that position into the order one pass over the list leaves
void pairs_to_edges_blocks(skb_ctx *c, unsigned long long *d_pairs, int64_t n_pairs, double min_af_pct,
                           unsigned long long sums[2], cudaEvent_t ev_mid, cudaEvent_t ev_end) {
    cudaEvent_t *ev = call_events(c);  // ev[3], ev[4] serve each block's pairs_to_edges (edge_call's -n stage comes after)
    CK(cudaEventRecord(ev_mid, c->st));
    const int32_t n = c->n();
    std::vector<int32_t> refs;
    if (n_pairs > 0) {
        PoolRef<uint8_t> d_mark(c->pool["table_blocks.mark"]);
        d_mark.reserve((size_t)n, 0, c->st);
        CK(cudaMemsetAsync(d_mark.p, 0, (size_t)n, c->st));
        launch(c, ref_mark_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, c->d_seed_off.p, d_pairs, n_pairs, (uint32_t)n,
               d_mark.p);
        std::vector<uint8_t> mark((size_t)n);
        CK(cudaMemcpyAsync(mark.data(), d_mark.p, (size_t)n, cudaMemcpyDeviceToHost, c->st));
        CK(cudaStreamSynchronize(c->st));
        for (int32_t g = 0; g < n; g++)
            if (mark[(size_t)g]) refs.push_back(g);
    }
    const std::vector<std::vector<int32_t>> blocks = table_blocks(c, refs);
    c->blocks_last_call = (int32_t)blocks.size();
    if (blocks.size() <= 1) {  // every pair in one block: nothing to select or merge
        if (!blocks.empty()) build_block_tables(c, blocks[0]);
        pairs_to_edges(c, d_pairs, blocks.empty() ? 0 : n_pairs, min_af_pct, sums, ev[3], ev_end);
        return;
    }
    if (n_pairs >= (1ll << 31)) throw CudaFail{"too many surviving pairs in one call"};  // as run_ani: 32-bit positions
    const bool det = c->ci || c->detailed;  // pairs_to_edges leaves a detail record per edge
    PoolRef<uint32_t> d_f(c->pool["table_blocks.flag"]), d_p(c->pool["table_blocks.pos"]);
    PoolRef<unsigned long long> d_sel(c->pool["table_blocks.pairs"]);
    PoolRef<uint32_t> d_sel_pos(c->pool["table_blocks.pair_pos"]), acc_pos(c->pool["table_blocks.edge_pos"]);
    PoolRef<skb_edge> acc(c->pool["table_blocks.edges"]);
    PoolRef<skb_edge_detail> acc_det(c->pool["table_blocks.detail"]);
    d_f.reserve((size_t)n_pairs + 1, 0, c->st);
    d_p.reserve((size_t)n_pairs + 1, 0, c->st);
    d_sel.reserve((size_t)n_pairs, 0, c->st);
    d_sel_pos.reserve((size_t)n_pairs, 0, c->st);
    int64_t total = 0;
    float ms_anchor = 0;
    int anchor_launches = 0;
    sums[0] = sums[1] = 0;
    for (const std::vector<int32_t> &blk : blocks) {
        build_block_tables(c, blk);
        launch(c, pair_owned_flag_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, c->d_seed_off.p, d_pairs, n_pairs,
               (uint32_t)n, (uint32_t)blk.front(), (uint32_t)blk.back() + 1, d_f.p);
        CK(cudaMemsetAsync(d_f.p + n_pairs, 0, 4, c->st));
        exclusive_scan_u32(c, d_f.p, d_p.p, (size_t)n_pairs + 1);
        launch(c, pair_keep_pos_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, d_pairs, n_pairs, d_f.p, d_p.p, d_sel.p,
               d_sel_pos.p);
        uint32_t m = 0;
        CK(cudaMemcpyAsync(&m, d_p.p + n_pairs, 4, cudaMemcpyDeviceToHost, c->st));
        CK(cudaStreamSynchronize(c->st));
        acc_pos.reserve((size_t)total + m, (size_t)total, c->st);  // the block's edges are at most its pairs
        unsigned long long s[2];
        pairs_to_edges(c, d_sel.p, m, min_af_pct, s, ev[3], ev[4], d_sel_pos.p, acc_pos.p + total);
        sums[0] += s[0];
        sums[1] += s[1];
        ms_anchor += c->last_ms_anchor;
        anchor_launches += c->last_anchor_launches;
        const int64_t ne = c->last_n_edges;
        if (ne) {
            acc.reserve((size_t)(total + ne), (size_t)total, c->st);
            CK(cudaMemcpyAsync(acc.p + total, c->last_dev_edges, (size_t)ne * sizeof(skb_edge), cudaMemcpyDeviceToDevice, c->st));
            if (det) {
                acc_det.reserve((size_t)(total + ne), (size_t)total, c->st);
                CK(cudaMemcpyAsync(acc_det.p + total, c->last_dev_detail, (size_t)ne * sizeof(skb_edge_detail),
                                   cudaMemcpyDeviceToDevice, c->st));
            }
        }
        total += ne;
    }
    PoolRef<skb_edge> merged(c->pool["table_blocks.merged"]);
    PoolRef<skb_edge_detail> merged_det(c->pool["table_blocks.merged_detail"]);
    if (total) {
        PoolRef<uint32_t> d_key_s(c->pool["table_blocks.pos_sorted"]);
        PoolRef<uint32_t> d_idx(c->pool["table_blocks.idx"]), d_perm(c->pool["table_blocks.perm"]);
        d_key_s.reserve((size_t)total, 0, c->st);
        d_idx.reserve((size_t)total, 0, c->st);
        d_perm.reserve((size_t)total, 0, c->st);
        merged.reserve((size_t)total, 0, c->st);
        launch(c, iota_u32_kernel, nblk((uint64_t)total, 256), 256, 0, total, d_idx.p);
        int pos_bits = 1;  // positions < n_pairs
        while (pos_bits < 32 && (1ll << pos_bits) < n_pairs) pos_bits++;
        sort_pairs(c, acc_pos.p, d_key_s.p, d_idx.p, d_perm.p, (size_t)total, pos_bits);
        launch(c, gather_kernel<skb_edge>, nblk((uint64_t)total, 256), 256, 0, acc.p, d_perm.p, total, merged.p);
        if (det) {
            merged_det.reserve((size_t)total, 0, c->st);
            launch(c, gather_kernel<skb_edge_detail>, nblk((uint64_t)total, 256), 256, 0, acc_det.p, d_perm.p, total,
                   merged_det.p);
        }
    }
    CK(cudaEventRecord(ev_end, c->st));
    CK(cudaEventSynchronize(ev_end));
    c->last_dev_edges = merged.p;
    c->last_dev_detail = det ? merged_det.p : nullptr;
    c->last_n_edges = total;
    c->last_ms_anchor = ms_anchor;
    c->last_anchor_launches = anchor_launches;
}

// skb_triangle, skb_pairs_edges and skb_rect after their argument checks: `pairs(EdgePairs &)` checks the context's state
// and leaves the pairs to evaluate (ms_screen), pairs_to_edges evaluates them (ms_ani), max_n > 0 cuts them to each
// query's best max_n (best_n_edges; its time counts in ms_total only), and the edges go to the caller -- a malloc'ed host
// copy when `edges` is given, the device copy in any case (skb_device_edges)
template <typename F>
int edge_call(skb_ctx *c, double min_af_pct, skb_edge **edges, int64_t *n_edges, skb_stats *stats, F &&pairs,
              int64_t max_n = 0) {
    // --ci is defined for the mean estimator only, and --detailed prints that interval too (DESIGN.md section 3)
    if ((c->ci || c->detailed) && c->estimator != SKB_ANI_MEAN)
        return fail(c, SKB_EINVAL, "the --ci interval and the --detailed columns are defined for the mean ANI estimator "
                                   "only (skb_set_ani_ci, skb_set_detailed, skb_set_ani_estimator)");
    const int64_t launches0 = c->launches;
    c->whole_triangle = -1;
    c->blocks_last_call = 0;
    cudaEvent_t *ev = call_events(c);
    CK(cudaEventRecord(ev[0], c->st));
    EdgePairs p;
    const int rc = pairs(p);
    if (rc != SKB_OK) return rc;
    unsigned long long sums[2];
    if (c->on_demand)
        pairs_to_edges_blocks(c, p.d_pairs, p.n, min_af_pct, sums, ev[1], ev[2]);
    else
        pairs_to_edges(c, p.d_pairs, p.n, min_af_pct, sums, ev[1], ev[2]);
    float ms_screen = 0, ms_ani = 0, ms_best_n = 0;
    CK(cudaEventElapsedTime(&ms_screen, ev[0], ev[1]));
    CK(cudaEventElapsedTime(&ms_ani, ev[1], ev[2]));
    if (max_n > 0 && c->last_n_edges > max_n) {  // fewer edges than max_n: no query has more
        CK(cudaEventRecord(ev[3], c->st));
        best_n_edges(c, max_n);
        CK(cudaEventRecord(ev[4], c->st));
        CK(cudaEventSynchronize(ev[4]));
        CK(cudaEventElapsedTime(&ms_best_n, ev[3], ev[4]));
    }
    const int64_t ne = c->last_n_edges;
    // rect lists are sorted by (ref, query) on the device already; nothing to do on the host
    if (edges) {
        skb_edge *h = (skb_edge *)std::malloc(std::max<size_t>(1, (size_t)ne) * sizeof(skb_edge));
        if (!h) throw CudaFail{"host out of memory for edges"};
        if (ne) {
            const cudaError_t e = cudaMemcpy(h, c->last_dev_edges, (size_t)ne * sizeof(skb_edge), cudaMemcpyDeviceToHost);
            if (e != cudaSuccess) {
                std::free(h);
                CK(e);
            }
        }
        *edges = h;
    }
    if (stats) {
        stats->n_pairs_total = p.total;
        stats->n_pairs_screened = p.n;
        stats->n_edges = ne;
        stats->ms_screen = ms_screen;
        stats->ms_ani = ms_ani;
        stats->ms_total = ms_screen + ms_ani + ms_best_n;
        stats->ms_anchor = c->last_ms_anchor;
        stats->n_anchor_launches = c->last_anchor_launches;
        stats->launches = c->launches - launches0;
        stats->sum_query_seeds = (int64_t)sums[0];
        stats->sum_anchors = (int64_t)sums[1];
    }
    *n_edges = ne;
    return SKB_OK;
}

// malloc'ed host copy of the `rec_bytes`-byte records the last edge call left on the device, one per edge, or nullptr
// when the host is out of memory (skb_last_edge_ci, skb_last_edge_detail)
void *last_edges_to_host(skb_ctx *c, const void *dev, size_t rec_bytes) {
    const size_t bytes = (size_t)c->last_n_edges * rec_bytes;
    void *h = std::malloc(std::max<size_t>(1, bytes));
    if (!h || !bytes) return h;
    cudaError_t e = cudaMemcpyAsync(h, dev, bytes, cudaMemcpyDeviceToHost, c->st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->st);
    if (e != cudaSuccess) {
        std::free(h);
        CK(e);
    }
    return h;
}

bool write_all(FILE *f, const void *p, size_t n) { return n == 0 || fwrite(p, 1, n, f) == n; }
bool read_all(FILE *f, void *p, size_t n) { return n == 0 || fread(p, 1, n, f) == n; }

}  // namespace

extern "C" {

void skb_default_params(skb_params *p) {
    p->min_contig_len = 500;
    p->chunk_len = 20000;
    p->band_bp = 2500;
    p->max_gap = 300;
    p->anchor_score = 20;
    p->min_anchors = 3;
    p->min_score = 45;
    p->max_mult = 8;
    p->max_chunk_chains = 8;
    p->ovl_num = 1;
    p->ovl_den = 2;
    p->span_ext = 170;
    p->debias_a = 1.438713;
    p->debias_g = 0.905292;
}

int skb_create(int32_t device, const skb_params *params, skb_ctx **out) {
    if (!out) return SKB_EINVAL;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) +
                         " (libskani_b200 has no CPU path)";
        return SKB_ECUDA;
    }
    if (device < 0 || device >= ndev) {
        g_create_error = "device index out of range";
        return SKB_EINVAL;
    }
    skb_ctx *c = new skb_ctx();
    c->device = device;
    if (params)
        c->prm = *params;
    else
        skb_default_params(&c->prm);
    const skb_params &p = c->prm;
    if (p.max_mult < 1 || p.max_mult > STAGE || (p.max_mult & (p.max_mult - 1)) || p.max_chunk_chains < 1 ||
        p.max_chunk_chains > SLOTS || p.band_bp >= (int32_t)CONTIG_PAD || p.band_bp < 1 || p.chunk_len < 64 ||
        p.chunk_len > 32767 || p.anchor_score < 1 || p.anchor_score > 20 || p.ovl_den < 1 || p.min_anchors < 1 ||
        p.min_score <= (p.min_anchors - 1) * p.anchor_score) {
        g_create_error = "parameter outside the range the kernels support";
        delete c;
        return SKB_EINVAL;
    }
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        g_create_error = std::string("CUDA init failed: ") + cudaGetErrorString(e);
        delete c;
        return SKB_ECUDA;
    }
    if (prop.major < 10) {
        g_create_error = std::string("device '") + prop.name + "' is not sm_100 class; this library is built for sm_100a only";
        delete c;
        return SKB_ECUDA;
    }
    c->sm_count = prop.multiProcessorCount;
    if (const char *e = std::getenv("SKB_TAB_X2")) {
        const int v = atoi(e);
        if (v == 1 || v == 2 || v == 4) c->tab_x2_forced = v;
    }
    *out = c;
    return SKB_OK;
}

void skb_destroy(skb_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (cudaEvent_t e : ctx->anchor_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : ctx->up_ev) cudaEventDestroy(e);
    if (ctx->st_copy) cudaStreamDestroy(ctx->st_copy);
    if (ctx->t0) cudaEventDestroy(ctx->t0);
    if (ctx->t1) cudaEventDestroy(ctx->t1);
    for (cudaEvent_t e : ctx->call_ev)
        if (e) cudaEventDestroy(e);
    for (char *p : ctx->h_matrix)
        if (p) cudaFreeHost(p);
    if (ctx->st) {
        cudaStreamSynchronize(ctx->st);
        cudaStreamDestroy(ctx->st);
    }
    delete ctx;
}

const char *skb_last_error(const skb_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
int32_t skb_n_genomes(const skb_ctx *ctx) { return ctx ? ctx->n() : 0; }
int skb_device_edges(skb_ctx *ctx, const skb_edge **dev_edges, int64_t *n_edges) {
    return guarded(ctx, [&]() -> int {
        if (!dev_edges || !n_edges) return fail(ctx, SKB_EINVAL, "bad arguments");
        *dev_edges = ctx->last_dev_edges;
        *n_edges = ctx->last_n_edges;
        return SKB_OK;
    });
}

int64_t skb_launch_count(const skb_ctx *ctx) { return ctx ? ctx->launches : 0; }
int skb_table_blocks(const skb_ctx *ctx, int32_t *on_demand, int32_t *blocks_last_call) {
    if (!ctx) return SKB_EINVAL;
    if (on_demand) *on_demand = ctx->on_demand ? 1 : 0;
    if (blocks_last_call) *blocks_last_call = ctx->blocks_last_call;
    return SKB_OK;
}
void *skb_stream(const skb_ctx *ctx) { return ctx ? (void *)ctx->st : nullptr; }
void skb_free(void *p) { std::free(p); }

static int clear_impl(skb_ctx *ctx, bool keep_tables) {
    return guarded(ctx, [&]() -> int {
        CK(cudaStreamSynchronize(ctx->st));
        ctx->genome_set++;
        ctx->db.clear();
        ctx->ix.clear();
        ctx->indexed = false;
        ctx->add_calls.clear();
        ctx->own_first = 0;
        ctx->own_count = -1;
        ctx->on_demand = false;
        ctx->block_budget = 0;
        if (!keep_tables) ctx->kept_n = 0;
        return SKB_OK;
    });
}

int skb_clear(skb_ctx *ctx) { return clear_impl(ctx, false); }
int skb_clear_keep_tables(skb_ctx *ctx) { return clear_impl(ctx, true); }

int skb_timer_start(skb_ctx *ctx) {
    return guarded(ctx, [&]() -> int {
        if (!ctx->t0) {
            CK(cudaEventCreate(&ctx->t0));
            CK(cudaEventCreate(&ctx->t1));
        }
        CK(cudaEventRecord(ctx->t0, ctx->st));
        return SKB_OK;
    });
}

int skb_timer_stop(skb_ctx *ctx, float *ms) {
    return guarded(ctx, [&]() -> int {
        if (!ctx->t0 || !ms) return fail(ctx, SKB_ESTATE, "timer not started");
        CK(cudaEventRecord(ctx->t1, ctx->st));
        CK(cudaEventSynchronize(ctx->t1));
        CK(cudaEventElapsedTime(ms, ctx->t0, ctx->t1));
        return SKB_OK;
    });
}

// skb_add_genomes (per_seq = false: one genome per packed file) and skb_add_sequences (per_seq: one per kept contig)
static int add_impl(skb_ctx *ctx, int32_t n, const skb_packed *const *genomes, bool per_seq) {
    return guarded(ctx, [&]() -> int {
        ctx->genome_set++;
        if (n < 0 || (n > 0 && !genomes)) return fail(ctx, SKB_EINVAL, "bad genome list");
        uint64_t n_new = per_seq ? 0 : (uint64_t)n;
        for (int32_t i = 0; i < n; i++) {
            const skb_packed *p = genomes[i];
            if (!p || !p->words || (p->n_words & 1) || p->n_words * 32 < p->n_bases || p->n_contigs < 0)
                return fail(ctx, SKB_EINVAL, "genome " + std::to_string(i) + ": malformed packed buffer");
            uint64_t s = 0;
            for (int32_t k = 0; k < p->n_contigs; k++) {
                s += (uint64_t)p->contig_lens[k];
                if (per_seq && p->contig_lens[k] <= 0) return fail(ctx, SKB_EINVAL, "empty contig");
                if (per_seq && (uint64_t)p->contig_lens[k] + CONTIG_PAD >= (1ull << 31))
                    return fail(ctx, SKB_ELIMIT, "sequence too large for 31-bit padded coordinates");
            }
            if (s != (uint64_t)p->n_bases) return fail(ctx, SKB_EINVAL, "contig lengths do not sum to n_bases");
            if (!per_seq && (uint64_t)p->n_bases + (uint64_t)p->n_contigs * CONTIG_PAD >= (1ull << 31))
                return fail(ctx, SKB_ELIMIT, "genome too large for 31-bit padded coordinates");
            if (per_seq && (uint64_t)p->n_bases >= (1ull << 32))  // a batch's seed and marker counts are 32-bit
                return fail(ctx, SKB_ELIMIT, "file too large for one sketch batch");
            if (per_seq) n_new += (uint64_t)p->n_contigs;
        }
        if ((uint64_t)ctx->n() + n_new >= GID_MASK) return fail(ctx, SKB_ELIMIT, "too many genomes (22-bit ids)");
        // batches of <= 1 Gi bases (per-batch seed/marker totals stay far below 2^32), grouped into
        // super-batches of <= 32 (8 GiB of packed words) whose H2D copies are all enqueued up front on a second stream: batch i+1
        // uploads while batch i is being sketched.
        ctx->add_calls.push_back({ctx->n(), ctx->db.n_mkeys});
        if (!ctx->st_copy) CK(cudaStreamCreateWithFlags(&ctx->st_copy, cudaStreamNonBlocking));
        PoolRef<uint64_t> d_packed(ctx->pool["add_genomes.d_packed"]);
        int32_t g0 = 0;
        while (g0 < n) {
            std::vector<int32_t> cut{g0};
            std::vector<uint64_t> woff{0};
            int32_t g = g0;
            while (g < n && cut.size() <= 32) {
                uint64_t bases = 0, words = 0;
                int32_t g1 = g;
                while (g1 < n && (g1 == g || bases + (uint64_t)genomes[g1]->n_bases <= (1ull << 30))) {
                    bases += (uint64_t)genomes[g1]->n_bases;
                    words += (uint64_t)genomes[g1]->n_words;
                    g1++;
                }
                cut.push_back(g1);
                woff.push_back(woff.back() + words);
                g = g1;
            }
            const size_t nbatch = cut.size() - 1;
            CK(cudaStreamSynchronize(ctx->st));  // previous users of the packed buffer are done
            d_packed.reserve(woff.back() + 2, 0, ctx->st);
            while (ctx->up_ev.size() < nbatch) {
                cudaEvent_t e;
                CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                ctx->up_ev.push_back(e);
            }
            static const bool trace = std::getenv("SKB_TRACE") != nullptr;  // diagnosis: upload/sketch timeline on stderr
            std::vector<cudaEvent_t> tev;
            auto mark = [&](cudaStream_t s) {
                if (!trace) return;
                cudaEvent_t e;
                CK(cudaEventCreate(&e));
                CK(cudaEventRecord(e, s));
                tev.push_back(e);
            };
            std::vector<BatchMeta> metas;
            for (size_t bi = 0; bi < nbatch; bi++)
                metas.push_back(sketch_meta(ctx, genomes, cut[bi], cut[bi + 1], d_packed.p + woff[bi], bi));
            mark(ctx->st_copy);
            for (size_t bi = 0; bi < nbatch; bi++) {
                uint64_t w = woff[bi];
                for (int32_t i = cut[bi]; i < cut[bi + 1];) {  // genomes adjacent in host memory go up as one copy
                    int32_t j = i + 1;
                    uint64_t words = (uint64_t)genomes[i]->n_words;
                    while (j < cut[bi + 1] && genomes[j]->words == genomes[i]->words + words) words += (uint64_t)genomes[j++]->n_words;
                    CK(cudaMemcpyAsync(d_packed.p + w, genomes[i]->words, (size_t)words * 8, cudaMemcpyHostToDevice,
                                       ctx->st_copy));
                    w += words;
                    i = j;
                }
                CK(cudaEventRecord(ctx->up_ev[bi], ctx->st_copy));
                mark(ctx->st_copy);
            }
            for (size_t bi = 0; bi < nbatch; bi++) {
                sketch_batch(ctx, genomes, cut[bi], cut[bi + 1], metas[bi], ctx->up_ev[bi], per_seq);
                mark(ctx->st);
            }
            if (trace) {
                CK(cudaDeviceSynchronize());
                for (size_t i = 1; i < tev.size(); i++) {
                    float ms = 0;
                    CK(cudaEventElapsedTime(&ms, tev[0], tev[i]));
                    fprintf(stderr, "[skb trace] add %s %zu done at %8.2f ms\n", i <= nbatch ? "copy  " : "sketch",
                            i <= nbatch ? i - 1 : i - 1 - nbatch, ms);
                }
                for (cudaEvent_t e : tev) cudaEventDestroy(e);
            }
            g0 = cut.back();
        }
        return SKB_OK;
    });
}

int skb_add_genomes(skb_ctx *ctx, int32_t n, const skb_packed *const *genomes) { return add_impl(ctx, n, genomes, false); }
int skb_add_sequences(skb_ctx *ctx, int32_t n_files, const skb_packed *const *files) {
    return add_impl(ctx, n_files, files, true);
}

// ---- the per-genome index -------------------------------------------------------------------------------------------
// Seed tables and chunk tables of the genomes [g0, n), laid out as anchor_kernel and the chain kernels read them
// (DESIGN.md §2): skb_index builds them with g0 = 0, skb_index_append for the genomes added since the last index.

// The sparsest seed tables the device holds comfortably: a lookup is one sector read unless its bucket overflowed, and
// at 0.5 records per bucket that is rare enough not to stall a warp (skb_probe.cuh).  SKB_TAB_X2 forces a density.
static int table_density(skb_ctx *c, uint64_t own_seeds) {
    // decided once per sketch-DB size: cudaMemGetInfo takes a driver-wide lock and stalls for tens of ms whenever a
    // monitoring tool (nvidia-smi / NVML polling) holds it -- seen as 20-80 ms spikes of this call
    if (!c->x2_decided || c->x2_decided_seeds != own_seeds) {
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const double budget = std::min(0.35 * (double)total_b,
                                       (double)free_b + (double)c->d_tab.cap * 8.0 - 40.0 * (double)(1ull << 30));
        c->x2_decided = 1;
        for (int x2 : {4, 2})
            if (((double)own_seeds * x2 / 2 + (double)c->n()) * BUCKET * 8.0 <= budget) {
                c->x2_decided = x2;
                break;
            }
        c->x2_decided_seeds = own_seeds;
        c->x2_budget = budget;
        c->x2_room = (double)free_b + (double)c->d_tab.cap * 8.0;
    }
    return c->tab_x2_forced ? c->tab_x2_forced : c->x2_decided;
}

// Seed tables and repeat flags of the genomes [g0, n) at density tab_x2.  Only the genomes this context owns get a
// table (skb_set_owned: the others are only ever queries here), so the tables of the owned genomes are laid out by
// those genomes in id order, their seed counts and the density alone: a rank builds its tables at ids 0..k-1 before
// the sketches are exchanged, and with `reuse` the tables already in d_tab serve the same genomes at own_first..
static int build_seed_tables(skb_ctx *c, int32_t g0, bool reuse) {
    const int32_t n = c->n();
    std::vector<uint64_t> &tab_off = c->ix.tab_off;
    std::vector<uint32_t> &buckets = c->ix.tab_buckets;
    tab_off.resize(n + 1);
    buckets.resize(n);
    for (int32_t g = g0; g < n; g++) {
        const uint64_t ns = c->db.seed_off[g + 1] - c->db.seed_off[g];
        if (ns >= (1ull << 31)) return fail(c, SKB_ELIMIT, "genome has too many seeds");
        buckets[g] = c->owns(g) ? table_buckets(c, g) : 0u;
        tab_off[g + 1] = tab_off[g] + (uint64_t)buckets[g] * BUCKET;
    }
    c->d_seed_off.upload(c->db.seed_off, g0, c->st);
    if (c->on_demand) {
        // the repeat flags of every genome (a query reads its own seeds' flags while only reference tables exist):
        // the tables are built block by block for them and dropped; edge calls build the ones they need again
        c->d_tab_off.reserve((size_t)n + 1, 0, c->st);
        c->d_tab_buckets.reserve((size_t)n, 0, c->st);
        std::vector<int32_t> ids(n - g0);
        for (int32_t g = g0; g < n; g++) ids[g - g0] = g;
        for (const std::vector<int32_t> &blk : table_blocks(c, ids)) build_block_tables(c, blk);
        CK(cudaStreamSynchronize(c->st));
        c->d_tab.release();  // the memory goes to the edge calls' blocks and their pair stage
        return SKB_OK;
    }
    c->d_tab_off.upload(tab_off, g0, c->st);
    c->d_tab_buckets.upload(buckets, g0, c->st);
    const uint64_t t0 = tab_off[g0], t1 = tab_off[n];
    c->d_tab.reserve(t1 + BUCKET, reuse ? t1 : t0, c->st);
    if (reuse) return SKB_OK;
    CK(cudaMemsetAsync(c->d_tab.p + t0, 0xFF, (t1 - t0) * 8, c->st));
    // the owned seeds are one contiguous range; the repeat flags of the others arrived with their seeds
    // (skb_import_sketches keeps them)
    const auto [o0, o1] = c->owned_in(g0, n);
    const uint64_t s0 = c->db.seed_off[o0], s1 = c->db.seed_off[o1];
    if (s1 > s0) {
        launch(c, tab_insert_kernel, nblk(s1 - s0, 256), 256, 0, c->d_seeds.p, s1, c->d_seed_off.p, n, c->d_tab.p,
               c->d_tab_off.p, c->d_tab_buckets.p, s0);
        launch(c, rep_flag_kernel, nblk(s1 - s0, 256), 256, 0, c->d_seeds.p, s1, c->d_seed_off.p, n, c->d_tab.p,
               c->d_tab_off.p, c->d_tab_buckets.p, c->prm.max_mult, s0);
    }
    return SKB_OK;
}

// Chunk tables of the genomes [g0, n): contigs in padded coordinates (CONTIG_PAD after each), cut into chunk_len
// pieces, and for every chunk (and one sentinel per genome) the index of its first seed.  Counted first, then filled
// in place, by a few host threads when the range is large (1.5 M chunks at config3: the push_back loop this replaced
// was 4 ms of every index build, and is replicated on every rank).
static int build_chunk_tables(skb_ctx *c, int32_t g0) {
    const int32_t n = c->n();
    const uint32_t CL = (uint32_t)c->prm.chunk_len;
    const skb_ctx::SketchDb &db = c->db;
    skb_ctx::HostIndex &ix = c->ix;
    ix.chunk_off.resize(n + 1);
    for (int32_t g = g0; g < n; g++) {
        uint64_t cnt = 0;
        for (uint32_t k = db.ctg_off[g]; k < db.ctg_off[g + 1]; k++) cnt += (db.ctg_len[k] + CL - 1) / CL;
        if ((uint64_t)ix.chunk_off[g] + cnt >= (1ull << 32)) return fail(c, SKB_ELIMIT, "too many chunks");
        ix.chunk_off[g + 1] = ix.chunk_off[g] + (uint32_t)cnt;
    }
    ix.ctg_pstart.resize(db.ctg_len.size());
    ix.chunk_start.resize(ix.chunk_off[n]);
    ix.chunk_len.resize(ix.chunk_off[n]);
    auto fill = [&](int32_t ga, int32_t gb) {
        for (int32_t g = ga; g < gb; g++) {
            uint32_t off = 0, at = ix.chunk_off[g];
            for (uint32_t k = db.ctg_off[g]; k < db.ctg_off[g + 1]; k++) {
                ix.ctg_pstart[k] = off;
                const uint32_t len = db.ctg_len[k];
                for (uint32_t st = 0; st < len; st += CL, at++) {
                    ix.chunk_start[at] = off + st;
                    ix.chunk_len[at] = std::min<uint32_t>(CL, len - st);
                }
                off += len + CONTIG_PAD;
            }
        }
    };
    const int64_t m = n - g0;
    const int n_thr = m >= 1024 ? 4 : 1;
    if (n_thr == 1)
        fill(g0, n);
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < n_thr; t++)
            pool.emplace_back(fill, g0 + (int32_t)(m * t / n_thr), g0 + (int32_t)(m * (t + 1) / n_thr));
        for (auto &th : pool) th.join();
    }
    const size_t k0 = db.ctg_off[g0], ch0 = ix.chunk_off[g0];
    c->d_total_len.upload(db.total_len, g0, c->st);
    c->d_ctg_off.upload(db.ctg_off, g0, c->st);
    c->d_ctg_len.upload(db.ctg_len, k0, c->st);
    c->d_ctg_pstart.upload(ix.ctg_pstart, k0, c->st);
    c->d_chunk_off.upload(ix.chunk_off, g0, c->st);
    c->d_chunk_start.upload(ix.chunk_start, ch0, c->st);
    c->d_chunk_len.upload(ix.chunk_len, ch0, c->st);
    const uint32_t e0 = (uint32_t)ch0 + (uint32_t)g0, e1 = ix.chunk_off[n] + (uint32_t)n;
    c->d_chunk_begin.reserve(e1, e0, c->st);
    launch(c, chunk_begin_kernel, nblk(e1 - e0, 256), 256, 0, c->d_seeds.p, c->d_seed_off.p, c->d_chunk_off.p, n,
           c->d_chunk_start.p, c->d_chunk_begin.p, e1, e0);
    return SKB_OK;
}

// Marker list offsets of the genomes [g0, n) from the per-genome counts the marker kernels left in d_marker_cnt
static void marker_offsets(skb_ctx *c, int32_t g0) {
    const int32_t n = c->n();
    std::vector<uint32_t> cnt((size_t)(n - g0));
    CK(cudaMemcpyAsync(cnt.data(), c->d_marker_cnt.p + g0, cnt.size() * 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    std::vector<uint64_t> &off = c->ix.marker_off;
    off.resize(n + 1);
    for (int32_t g = g0; g < n; g++) off[g + 1] = off[g] + cnt[(size_t)(g - g0)];
    c->d_marker_off.upload(off, g0, c->st);
    CK(cudaStreamSynchronize(c->st));
}

int skb_index(skb_ctx *ctx) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        static const bool trace = std::getenv("SKB_TRACE") != nullptr;  // diagnosis: phase times on stderr (adds syncs)
        double t_last = 0;
        auto lap = [&](const char *what) {
            if (!trace) return;
            cudaStreamSynchronize(c->st);
            timespec ts;
            clock_gettime(CLOCK_MONOTONIC, &ts);
            const double now = ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
            if (what) fprintf(stderr, "[skb trace] index %-14s %7.2f ms\n", what, now - t_last);
            t_last = now;
        };
        lap(nullptr);
        const int32_t n = c->n();
        if (n == 0) return fail(c, SKB_ESTATE, "no genomes added");
        const auto [o0, o1] = c->owned_in(0, n);
        const uint64_t own_seeds = c->db.seed_off[o1] - c->db.seed_off[o0];
        // tables of exactly the owned genomes are already in d_tab (built before the sketches were exchanged)
        const bool reuse = c->kept_n > 0 && c->kept_n == o1 - o0 && c->kept_seeds == own_seeds;
        c->tab_x2 = reuse ? c->kept_x2 : table_density(c, own_seeds);
        // on-demand tables when the tables at that density, sized as table_density sizes them, exceed the budget; a
        // context that owns part of the tables (skb_set_owned) keeps them resident
        c->on_demand = !reuse && c->own_count < 0 &&
                       ((double)own_seeds * c->tab_x2 / 2 + (double)n) * BUCKET * 8.0 > table_budget(c);
        c->block_budget = 0;  // measured for the repeat flags' blocks now, and again by the first edge call (below)
        int rc = build_seed_tables(c, 0, reuse);
        if (rc != SKB_OK) return rc;
        c->kept_n = 0;
        lap("seed tables");
        if ((rc = build_chunk_tables(c, 0)) != SKB_OK) return rc;
        lap("chunk tables");
        // ---- markers: sort raw keys, unique -> inverted index; per-genome counts; per-genome lists
        c->d_marker_cnt.reserve((size_t)n, 0, c->st);
        CK(cudaMemsetAsync(c->d_marker_cnt.p, 0, (size_t)n * 4, c->st));
        c->ix.n_inv = 0;
        const uint64_t nk = c->db.n_mkeys;
        if (nk) {
            if (nk >= (1ull << 32)) return fail(c, SKB_ELIMIT, "too many marker keys");
            PoolRef<uint64_t> d_sorted(c->pool["skb_index.d_sorted"]);
            PoolRef<uint32_t> d_flag(c->pool["skb_index.d_flag"]), d_pos(c->pool["skb_index.d_pos"]);
            d_sorted.reserve(nk, 0, c->st);
            d_flag.reserve(nk + 1, 0, c->st);
            d_pos.reserve(nk + 1, 0, c->st);
            // raw keys arrive genome by genome (ids ascending: skb_add_genomes, skb_import_sketches, skb_db_load), so a
            // STABLE sort on the 42 marker bits alone leaves every marker's run ordered by genome id: 6 radix passes
            // instead of 8
            sort_keys_u64(c, c->d_mkeys.p, d_sorted.p, nk, 64, GID_BITS);
            launch(c, unique_flag_kernel, nblk(nk, 256), 256, 0, d_sorted.p, nk, d_flag.p);
            CK(cudaMemsetAsync(d_flag.p + nk, 0, 4, c->st));
            exclusive_scan_u32(c, d_flag.p, d_pos.p, nk + 1);
            uint32_t nu = 0;
            CK(cudaMemcpyAsync(&nu, d_pos.p + nk, 4, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            c->ix.n_inv = nu;
            c->d_inv.reserve(nu + 1, 0, c->st);
            launch(c, unique_scatter_kernel, nblk(nk, 256), 256, 0, d_sorted.p, nk, d_flag.p, d_pos.p, c->d_inv.p,
                   c->d_marker_cnt.p);
            lap("inverted index");
            // per-genome sorted lists: swap key halves, sort again, strip ids
            c->d_markers.reserve(nu + 1, 0, c->st);
            launch(c, swap_key_kernel, nblk(nu, 256), 256, 0, c->d_inv.p, nu, d_sorted.p);
            // the input is ordered by marker: a stable sort on the 22 genome bits alone keeps each genome's markers
            // ascending (3 passes instead of 8)
            sort_keys_u64(c, d_sorted.p, c->d_markers.p, nu, 64, 2 * K_MARKER);
            launch(c, strip_gid_kernel, nblk(nu, 256), 256, 0, c->d_markers.p, nu);
        }
        marker_offsets(c, 0);
        lap("marker lists");
        c->ix.n_indexed = n;
        c->ix.n_inv_genomes = n;
        c->ix.n_mkeys_indexed = nk;
        c->block_budget = 0;  // the marker sort's scratch is allocated now
        c->indexed = true;
        return SKB_OK;
    });
}

// Seed tables and repeat flags of the genomes added so far, nothing else: the first half of skb_index, for a rank that is
// about to exchange sketches.  With skb_clear_keep_tables the tables survive the exchange, and the skb_index that follows
// (after skb_import_sketches + skb_set_owned for the same genomes) reuses them instead of building them again.
int skb_index_seed_tables(skb_ctx *ctx) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        const int32_t n = c->n();
        if (n == 0) return fail(c, SKB_ESTATE, "no genomes added");
        const auto [o0, o1] = c->owned_in(0, n);
        const uint64_t own_seeds = c->db.seed_off[o1] - c->db.seed_off[o0];
        c->tab_x2 = table_density(c, own_seeds);
        c->on_demand = false;
        const int rc = build_seed_tables(c, 0, false);
        if (rc != SKB_OK) return rc;
        CK(cudaStreamSynchronize(c->st));
        c->kept_n = o1 - o0;
        c->kept_seeds = own_seeds;
        c->kept_x2 = c->tab_x2;
        c->indexed = false;
        return SKB_OK;
    });
}

// Index the genomes added since the last skb_index / skb_index_append as QUERY-ONLY additions: their
// seed tables (at the density of the last skb_index), repeat flags, chunk tables and sorted marker lists are appended;
// the inverted marker index is left alone (they can be the query side of skb_rect, not a reference, and not part of a
// triangle).  This is what `skani search` needs: the database stays resident and indexed, one query
// genome comes and goes (skb_pop_last_add) at the cost of its own sketch.
int skb_index_append(skb_ctx *ctx) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        const int32_t n = c->n(), n0 = c->ix.n_indexed;
        if (!c->indexed && n0 == 0) return fail(c, SKB_ESTATE, "call skb_index on the database first");
        if (n == n0) {
            c->indexed = true;
            return SKB_OK;
        }
        int rc = build_seed_tables(c, n0, false);
        if (rc != SKB_OK) return rc;
        if ((rc = build_chunk_tables(c, n0)) != SKB_OK) return rc;
        // sorted unique marker lists of the new genomes, appended behind the database's
        const uint64_t nk = c->db.n_mkeys - c->ix.n_mkeys_indexed;
        c->d_marker_cnt.reserve((size_t)n, (size_t)n0, c->st);
        CK(cudaMemsetAsync(c->d_marker_cnt.p + n0, 0, (size_t)(n - n0) * 4, c->st));
        if (nk) {
            PoolRef<uint64_t> d_a(c->pool["skb_index_append.a"]), d_b(c->pool["skb_index_append.b"]);
            PoolRef<uint32_t> d_flag(c->pool["skb_index_append.flag"]), d_pos(c->pool["skb_index_append.pos"]);
            d_a.reserve(nk, 0, c->st);
            d_b.reserve(nk, 0, c->st);
            d_flag.reserve(nk + 1, 0, c->st);
            d_pos.reserve(nk + 1, 0, c->st);
            launch(c, swap_key_kernel, nblk(nk, 256), 256, 0, c->d_mkeys.p + c->ix.n_mkeys_indexed, nk, d_a.p);
            sort_keys_u64(c, d_a.p, d_b.p, nk);
            launch(c, unique_flag_kernel, nblk(nk, 256), 256, 0, d_b.p, nk, d_flag.p);
            CK(cudaMemsetAsync(d_flag.p + nk, 0, 4, c->st));
            exclusive_scan_u32(c, d_flag.p, d_pos.p, nk + 1);
            uint32_t nu = 0;
            CK(cudaMemcpyAsync(&nu, d_pos.p + nk, 4, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            const uint64_t m0 = c->ix.marker_off[n0];
            c->d_markers.reserve(m0 + nu + 1, m0, c->st);
            launch(c, unique_scatter_swapped_kernel, nblk(nk, 256), 256, 0, d_b.p, nk, d_flag.p, d_pos.p, c->d_markers.p + m0,
                   c->d_marker_cnt.p);
        }
        marker_offsets(c, n0);
        c->ix.n_mkeys_indexed = c->db.n_mkeys;
        c->ix.n_indexed = n;
        c->indexed = true;
        return SKB_OK;
    });
}

// Undo the most recent skb_add_genomes / skb_add_sequences call (and its index entries): the query genomes of a search leave.
int skb_pop_last_add(skb_ctx *ctx) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (c->add_calls.empty()) return fail(c, SKB_ESTATE, "nothing to pop");
        const skb_ctx::AddCall a = c->add_calls.back();
        if (a.n_before < c->ix.n_inv_genomes) return fail(c, SKB_ESTATE, "cannot pop genomes that are part of the inverted index");
        CK(cudaStreamSynchronize(c->st));
        c->genome_set++;
        c->add_calls.pop_back();
        c->db.truncate(a.n_before, a.mkeys_before);
        c->ix.truncate(c->db);
        c->indexed = c->ix.n_indexed == a.n_before && a.n_before > 0;
        return SKB_OK;
    });
}

int skb_sketch_sizes(skb_ctx *ctx, int32_t g, int64_t *n_seeds, int64_t *n_markers, int32_t *n_chunks,
                     int64_t *total_len) {
    if (!ctx) return SKB_EINVAL;
    if (g < 0 || g >= ctx->n()) return fail(ctx, SKB_EINVAL, "genome id out of range");
    if (n_seeds) *n_seeds = (int64_t)(ctx->db.seed_off[g + 1] - ctx->db.seed_off[g]);
    if (total_len) *total_len = (int64_t)ctx->db.total_len[g];
    if (n_markers || n_chunks) {
        if (!ctx->indexed || g >= ctx->ix.n_indexed) return fail(ctx, SKB_ESTATE, "call skb_index first");
        if (n_markers) *n_markers = (int64_t)(ctx->ix.marker_off[g + 1] - ctx->ix.marker_off[g]);
        if (n_chunks) *n_chunks = (int32_t)(ctx->ix.chunk_off[g + 1] - ctx->ix.chunk_off[g]);
    }
    return SKB_OK;
}

int skb_get_seeds(skb_ctx *ctx, int32_t g, uint64_t *out) {
    return guarded(ctx, [&]() -> int {
        if (g < 0 || g >= ctx->n() || !out) return fail(ctx, SKB_EINVAL, "bad arguments");
        const uint64_t a = ctx->db.seed_off[g], b = ctx->db.seed_off[g + 1];
        CK(cudaStreamSynchronize(ctx->st));
        if (b > a) CK(cudaMemcpy(out, ctx->d_seeds.p + a, (b - a) * 8, cudaMemcpyDeviceToHost));
        return SKB_OK;
    });
}

int skb_get_markers(skb_ctx *ctx, int32_t g, uint64_t *out) {
    return guarded(ctx, [&]() -> int {
        if (!ctx->indexed || g < 0 || g >= ctx->ix.n_indexed || !out) return fail(ctx, SKB_ESTATE, "not indexed / bad id");
        const uint64_t a = ctx->ix.marker_off[g], b = ctx->ix.marker_off[g + 1];
        CK(cudaStreamSynchronize(ctx->st));
        if (b > a) CK(cudaMemcpy(out, ctx->d_markers.p + a, (b - a) * 8, cudaMemcpyDeviceToHost));
        return SKB_OK;
    });
}

// Marker prescreen of this partition's rows of the triangle; leaves the surviving pairs (a << 32 | b, a < b, sorted)
// on the device.  Rows of the dense count matrix are processed in tiles that fit a memory budget, so the matrix
// never has to hold rows x n counters at once (n = 50,000: 10 GB).
static int screen_triangle_impl(skb_ctx *c, double screen_pct, int32_t part, int32_t n_parts, EdgePairs &out) {
    if (n_parts < 1 || part < 0 || part >= n_parts) return fail(c, SKB_EINVAL, "bad arguments");
    if (!c->indexed || c->ix.n_indexed != c->n()) return fail(c, SKB_ESTATE, "call skb_index first");
    if (c->ix.n_inv_genomes != c->n()) return fail(c, SKB_ESTATE, "query-only genomes present: triangle needs skb_index");
    const uint32_t n = (uint32_t)c->ix.n_indexed;
    const uint32_t rows_local = rows_owned(n, (uint32_t)part, (uint32_t)n_parts);
    int64_t pairs_total = 0;
    for (uint32_t rl = 0; rl < rows_local; rl++) pairs_total += n - 1 - row_global(rl, (uint32_t)part, (uint32_t)n_parts);
    out.total = pairs_total;
    PoolRef<uint32_t> d_cnt(c->pool["skb_triangle.d_cnt"]);
    PoolRef<unsigned long long> d_pairs(c->pool["skb_triangle.d_pairs"]), d_pairs_sorted(c->pool["skb_triangle.d_pairs_sorted"]), d_np(c->pool["skb_triangle.d_np"]);
    d_np.reserve(1, 0, c->st);
    const double scale = screen_pct > 0.0 ? std::pow(screen_pct / 100.0, (double)K_MARKER) : 0.0;
    static const uint64_t tile_bytes = [] {
        const char *e = std::getenv("SKB_SCREEN_TILE_MB");
        return (uint64_t)(e ? std::max(1, atoi(e)) : 2048) << 20;
    }();
    const uint32_t tile_rows = (uint32_t)std::max<uint64_t>(2, std::min<uint64_t>(rows_local, tile_bytes / (4ull * std::max(n, 1u)))) & ~1u;
    unsigned long long np = 0;
    std::vector<unsigned long long> tile_np;
    // pass 1 per tile: count survivors (the count matrix is rebuilt per tile in pass 2; run counting is cheap)
    for (int pass = 0; pass < 2; pass++) {
        unsigned long long at = 0;
        size_t ti = 0;
        if (pass == 1) {
            if (!np) break;
            d_pairs.reserve(np, 0, c->st);
            d_pairs_sorted.reserve(np, 0, c->st);
        }
        for (uint32_t r0 = 0; r0 < rows_local; r0 += tile_rows, ti++) {
            const uint32_t nr = std::min(tile_rows, rows_local - r0);
            const uint64_t cells = (uint64_t)nr * n;
            if (pass == 1 && tile_np[ti] == 0) continue;
            if (pass == 0 || rows_local > tile_rows) {  // a single tile keeps its counts from pass 0
                d_cnt.reserve(cells, 0, c->st);
                if (scale > 0.0) {
                    CK(cudaMemsetAsync(d_cnt.p, 0, cells * 4, c->st));
                    if (c->ix.n_inv)
                        launch(c, screen_runs_kernel, nblk(c->ix.n_inv, 256), 256, 0, c->d_inv.p, c->ix.n_inv, d_cnt.p, n, part,
                               n_parts, r0, nr);
                }
            }
            CK(cudaMemsetAsync(d_np.p, 0, 8, c->st));
            launch(c, screen_compact_kernel, nblk(cells, 256), 256, 0, d_cnt.p, n, nr, r0, part, n_parts, c->d_marker_cnt.p,
                   scale, pass ? d_pairs.p + at : nullptr, d_np.p, pass ? tile_np[ti] : 0ull);
            if (pass == 0) {
                unsigned long long t = 0;
                CK(cudaMemcpyAsync(&t, d_np.p, 8, cudaMemcpyDeviceToHost, c->st));
                CK(cudaStreamSynchronize(c->st));
                tile_np.push_back(t);
                np += t;
            } else
                at += tile_np[ti];
        }
    }
    if (np) sort_keys_u64(c, (const uint64_t *)d_pairs.p, (uint64_t *)d_pairs_sorted.p, np);
    out.d_pairs = d_pairs_sorted.p;
    out.n = (int64_t)np;
    return SKB_OK;
}

int skb_triangle(skb_ctx *ctx, double screen_pct, double min_af_pct, int32_t part, int32_t n_parts,
                 skb_edge **edges, int64_t *n_edges, skb_stats *stats) {
    return guarded(ctx, [&]() -> int {
        if (!n_edges) return fail(ctx, SKB_EINVAL, "bad arguments");
        const int rc = edge_call(ctx, min_af_pct, edges, n_edges, stats,
                                 [&](EdgePairs &p) { return screen_triangle_impl(ctx, screen_pct, part, n_parts, p); });
        if (rc == SKB_OK && n_parts == 1) ctx->whole_triangle = (int64_t)ctx->genome_set;
        return rc;
    });
}

// ---- the triangle in two steps, for callers that exchange the surviving pairs between GPUs in between
// (skder_b200/multi.py: every rank screens its rows, the pair lists are all-gathered, every rank evaluates the pairs
// whose REFERENCE genome it owns -- the only seed tables it has built, skb_set_owned)
int skb_set_owned(skb_ctx *ctx, int32_t first, int32_t count) {
    return guarded(ctx, [&]() -> int {
        if (first < 0 || count < -1) return fail(ctx, SKB_EINVAL, "bad owned range");
        ctx->own_first = first;
        ctx->own_count = count;
        ctx->indexed = false;
        return SKB_OK;
    });
}

int skb_screen_triangle(skb_ctx *ctx, double screen_pct, int32_t part, int32_t n_parts, const uint64_t **dev_pairs,
                        int64_t *n_pairs, skb_stats *stats) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!dev_pairs || !n_pairs) return fail(c, SKB_EINVAL, "bad arguments");
        const int64_t launches0 = c->launches;
        cudaEvent_t *ev = call_events(c);
        CK(cudaEventRecord(ev[0], c->st));
        EdgePairs p;
        const int rc = screen_triangle_impl(c, screen_pct, part, n_parts, p);
        if (rc != SKB_OK) return rc;
        CK(cudaEventRecord(ev[1], c->st));
        CK(cudaEventSynchronize(ev[1]));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ev[0], ev[1]));
        *dev_pairs = (const uint64_t *)p.d_pairs;
        *n_pairs = p.n;
        if (stats) {
            std::memset(stats, 0, sizeof(*stats));
            stats->n_pairs_total = p.total;
            stats->n_pairs_screened = p.n;
            stats->ms_screen = stats->ms_total = ms;
            stats->launches = c->launches - launches0;
        }
        return SKB_OK;
    });
}

int skb_pairs_edges(skb_ctx *ctx, const uint64_t *dev_pairs, int64_t n_pairs, int32_t owned_only, double min_af_pct,
                    skb_edge **edges, int64_t *n_edges, skb_stats *stats) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!n_edges || n_pairs < 0 || (n_pairs && !dev_pairs)) return fail(c, SKB_EINVAL, "bad arguments");
        return edge_call(c, min_af_pct, edges, n_edges, stats, [&](EdgePairs &p) -> int {
            if (!c->indexed || c->ix.n_indexed != c->n()) return fail(c, SKB_ESTATE, "call skb_index first");
            p.d_pairs = (unsigned long long *)dev_pairs;
            p.n = p.total = n_pairs;
            if (n_pairs && (owned_only || c->own_count >= 0)) {
                // keep the pairs whose reference genome (more seeds; ties: b) this context owns, order preserved
                PoolRef<uint32_t> d_f(c->pool["pairs_edges.flag"]), d_p(c->pool["pairs_edges.pos"]);
                PoolRef<unsigned long long> d_keep(c->pool["pairs_edges.keep"]);
                d_f.reserve((size_t)n_pairs + 1, 0, c->st);
                d_p.reserve((size_t)n_pairs + 1, 0, c->st);
                d_keep.reserve((size_t)n_pairs, 0, c->st);
                const int32_t o0 = c->own_count < 0 ? 0 : c->own_first, o1 = c->own_count < 0 ? c->n() : c->own_first + c->own_count;
                launch(c, pair_owned_flag_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, c->d_seed_off.p, p.d_pairs, n_pairs,
                       (uint32_t)c->n(), (uint32_t)o0, (uint32_t)o1, d_f.p);
                CK(cudaMemsetAsync(d_f.p + n_pairs, 0, 4, c->st));
                exclusive_scan_u32(c, d_f.p, d_p.p, (size_t)n_pairs + 1);
                launch(c, pair_keep_kernel, nblk((uint64_t)n_pairs, 256), 256, 0, p.d_pairs, n_pairs, d_f.p, d_p.p, d_keep.p);
                uint32_t kept = 0;
                CK(cudaMemcpyAsync(&kept, d_p.p + n_pairs, 4, cudaMemcpyDeviceToHost, c->st));
                CK(cudaStreamSynchronize(c->st));
                p.d_pairs = d_keep.p;
                p.n = kept;
            }
            return SKB_OK;
        });
    });
}

// Marker prescreen of the rectangle refs x queries; leaves the surviving pairs (ref << 32 | query, sorted) on the device
static int screen_rect_impl(skb_ctx *c, const int32_t *refs, int32_t n_refs, const int32_t *queries, int32_t n_queries,
                            double screen_pct, EdgePairs &out) {
    if (!c->indexed || c->ix.n_indexed != c->n()) return fail(c, SKB_ESTATE, "call skb_index first");
    if (c->own_count >= 0) return fail(c, SKB_ESTATE, "skb_rect on a context that owns only part of the seed tables (skb_set_owned)");
    const int32_t n = c->ix.n_indexed;
    std::vector<int32_t> ref_slot(n, -1);
    for (int32_t i = 0; i < n_refs; i++) {
        if (refs[i] < 0 || refs[i] >= n) return fail(c, SKB_EINVAL, "reference id out of range");
        if (refs[i] >= c->ix.n_inv_genomes && screen_pct > 0.0)
            return fail(c, SKB_ESTATE, "a query-only genome (skb_index_append) cannot be a screened reference");
        if (ref_slot[refs[i]] >= 0) return fail(c, SKB_EINVAL, "duplicate reference id");
        ref_slot[refs[i]] = i;
    }
    std::vector<uint64_t> qpref(n_queries + 1, 0);
    for (int32_t i = 0; i < n_queries; i++) {
        if (queries[i] < 0 || queries[i] >= n) return fail(c, SKB_EINVAL, "query id out of range");
        qpref[i + 1] = qpref[i] + (c->ix.marker_off[queries[i] + 1] - c->ix.marker_off[queries[i]]);
    }
    PoolRef<int32_t> d_refs(c->pool["skb_rect.d_refs"]), d_queries(c->pool["skb_rect.d_queries"]), d_slot(c->pool["skb_rect.d_slot"]);
    PoolRef<uint64_t> d_qpref(c->pool["skb_rect.d_qpref"]);
    PoolRef<uint32_t> d_cnt(c->pool["skb_rect.d_cnt"]);
    PoolRef<unsigned long long> d_pairs(c->pool["skb_rect.d_pairs"]), d_pairs_sorted(c->pool["skb_rect.d_pairs_sorted"]), d_np(c->pool["skb_rect.d_np"]);
    const uint64_t cells = (uint64_t)n_refs * (uint64_t)n_queries;
    unsigned long long np = 0;
    d_np.reserve(1, 0, c->st);
    CK(cudaMemsetAsync(d_np.p, 0, 8, c->st));
    const double scale = screen_pct > 0.0 ? std::pow(screen_pct / 100.0, (double)K_MARKER) : 0.0;
    if (cells) {
        d_refs.upload(std::vector<int32_t>(refs, refs + n_refs), c->st);
        d_queries.upload(std::vector<int32_t>(queries, queries + n_queries), c->st);
        d_slot.upload(ref_slot, c->st);
        d_qpref.upload(qpref, c->st);
        d_cnt.reserve(cells, 0, c->st);
        if (scale > 0.0) {
            CK(cudaMemsetAsync(d_cnt.p, 0, cells * 4, c->st));
            if (qpref[n_queries] && c->ix.n_inv)
                launch(c, screen_rect_kernel, nblk(qpref[n_queries], 256), 256, 0, c->d_inv.p, c->ix.n_inv, c->d_markers.p,
                       c->d_marker_off.p, d_queries.p, n_queries, d_qpref.p, d_slot.p, d_cnt.p, (uint32_t)n_refs);
        }
        launch(c, screen_rect_compact_kernel, nblk(cells, 256), 256, 0, d_cnt.p, d_refs.p, (uint32_t)n_refs, d_queries.p,
               (uint32_t)n_queries, c->d_marker_cnt.p, scale, nullptr, d_np.p, 0ull);
        CK(cudaMemcpyAsync(&np, d_np.p, 8, cudaMemcpyDeviceToHost, c->st));
        CK(cudaStreamSynchronize(c->st));
        if (np) {
            d_pairs.reserve(np, 0, c->st);
            d_pairs_sorted.reserve(np, 0, c->st);
            CK(cudaMemsetAsync(d_np.p, 0, 8, c->st));
            launch(c, screen_rect_compact_kernel, nblk(cells, 256), 256, 0, d_cnt.p, d_refs.p, (uint32_t)n_refs, d_queries.p,
                   (uint32_t)n_queries, c->d_marker_cnt.p, scale, d_pairs.p, d_np.p, np);
            sort_keys_u64(c, (const uint64_t *)d_pairs.p, (uint64_t *)d_pairs_sorted.p, np);
        }
    }
    out.d_pairs = d_pairs_sorted.p;
    out.n = (int64_t)np;
    out.total = (int64_t)cells;
    return SKB_OK;
}

int skb_rect(skb_ctx *ctx, const int32_t *refs, int32_t n_refs, const int32_t *queries, int32_t n_queries,
             double screen_pct, double min_af_pct, skb_edge **edges, int64_t *n_edges, skb_stats *stats) {
    return guarded(ctx, [&]() -> int {
        if (!edges || !n_edges || n_refs < 0 || n_queries < 0 || (n_refs && !refs) || (n_queries && !queries))
            return fail(ctx, SKB_EINVAL, "bad arguments");
        return edge_call(
            ctx, min_af_pct, edges, n_edges, stats,
            [&](EdgePairs &p) { return screen_rect_impl(ctx, refs, n_refs, queries, n_queries, screen_pct, p); },
            ctx->max_results);
    });
}

int skb_set_ani_estimator(skb_ctx *ctx, int32_t estimator) {
    return guarded(ctx, [&]() -> int {
        if (estimator != SKB_ANI_MEAN && estimator != SKB_ANI_MEDIAN && estimator != SKB_ANI_ROBUST)
            return fail(ctx, SKB_EINVAL, "unknown ANI estimator " + std::to_string(estimator));
        ctx->estimator = estimator;
        return SKB_OK;
    });
}

int skb_set_ani_ci(skb_ctx *ctx, int32_t enabled) {
    return guarded(ctx, [&]() -> int {
        ctx->ci = enabled != 0;
        return SKB_OK;
    });
}

int skb_last_edge_ci(skb_ctx *ctx, double **lo_hi, int64_t *n) {
    return guarded(ctx, [&]() -> int {
        if (!lo_hi || !n) return fail(ctx, SKB_EINVAL, "bad arguments");
        if (!ctx->last_ci)
            return fail(ctx, SKB_ESTATE, "the last skb_triangle / skb_rect / skb_pairs_edges call ran without --ci (skb_set_ani_ci)");
        // the interval is the one --detailed prints: gathered from the same records, 16 of their 48 bytes copied
        const int64_t ne = ctx->last_n_edges;
        PoolRef<double2> d_lo_hi(ctx->pool["ci.lo_hi"]);
        if (ne) {
            d_lo_hi.reserve((size_t)ne, 0, ctx->st);
            launch(ctx, detail_ci_gather_kernel, nblk((uint64_t)ne, 256), 256, 0, ctx->last_dev_detail, ne, d_lo_hi.p);
        }
        double *h = (double *)last_edges_to_host(ctx, d_lo_hi.p, sizeof(double2));
        if (!h) return fail(ctx, SKB_ENOMEM, "host out of memory for the intervals");
        *lo_hi = h;
        *n = ne;
        return SKB_OK;
    });
}

int skb_set_detailed(skb_ctx *ctx, int32_t enabled) {
    return guarded(ctx, [&]() -> int {
        ctx->detailed = enabled != 0;
        return SKB_OK;
    });
}

int skb_set_max_results(skb_ctx *ctx, int64_t n) {
    return guarded(ctx, [&]() -> int {
        if (n < 0) return fail(ctx, SKB_EINVAL, "the number of results per query must be at least 0 (0: all)");
        ctx->max_results = n;
        return SKB_OK;
    });
}

int skb_set_marker_compression(skb_ctx *ctx, int64_t m) {
    return guarded(ctx, [&]() -> int {
        if (m < 1) return fail(ctx, SKB_EINVAL, "marker compression must be at least 1");
        if ((uint64_t)m == ctx->marker_c) return SKB_OK;
        // every genome of a context is sketched at one density: the screen compares marker counts across genomes
        if (ctx->n() != 0) return fail(ctx, SKB_ESTATE, "context already holds genomes sketched at another marker compression");
        ctx->marker_c = (uint64_t)m;
        return SKB_OK;
    });
}

int skb_marker_compression(const skb_ctx *ctx, int64_t *m) {
    if (!ctx || !m) return SKB_EINVAL;
    *m = (int64_t)ctx->marker_c;
    return SKB_OK;
}

int skb_last_edge_detail(skb_ctx *ctx, skb_edge_detail **out, int64_t *n) {
    return guarded(ctx, [&]() -> int {
        if (!out || !n) return fail(ctx, SKB_EINVAL, "bad arguments");
        if (!ctx->last_detailed)
            return fail(ctx, SKB_ESTATE,
                        "the last skb_triangle / skb_rect / skb_pairs_edges call ran without --detailed (skb_set_detailed)");
        skb_edge_detail *h = (skb_edge_detail *)last_edges_to_host(ctx, ctx->last_dev_detail, sizeof(skb_edge_detail));
        if (!h) return fail(ctx, SKB_ENOMEM, "host out of memory for the edge details");
        *out = h;
        *n = ctx->last_n_edges;
        return SKB_OK;
    });
}

int skb_genome_contig_stats(skb_ctx *ctx, int32_t first, int32_t n, int32_t *n_contigs, int64_t *nx) {
    return guarded(ctx, [&]() -> int {
        if (n < 0 || first < 0 || first > ctx->n() - n || (n && (!n_contigs || !nx))) return fail(ctx, SKB_EINVAL, "bad arguments");
        const skb_ctx::SketchDb &db = ctx->db;
        std::vector<uint32_t> len;
        for (int32_t i = 0; i < n; i++) {
            const int32_t g = first + i;
            len.assign(db.ctg_len.begin() + db.ctg_off[g], db.ctg_len.begin() + db.ctg_off[g + 1]);
            std::sort(len.begin(), len.end(), std::greater<uint32_t>());
            uint64_t total = 0;
            for (uint32_t l : len) total += l;
            // Nx: the length l_k of the first k (lengths descending) with 100 (l_1 + ... + l_k) >= x T
            const int xs[3] = {90, 50, 10};
            for (int j = 0; j < 3; j++) {
                uint64_t cum = 0;
                int64_t v = 0;
                for (uint32_t l : len) {
                    cum += l;
                    if (100 * cum >= (uint64_t)xs[j] * total) {
                        v = l;
                        break;
                    }
                }
                nx[3 * (size_t)i + j] = v;
            }
            n_contigs[i] = (int32_t)len.size();
        }
        return SKB_OK;
    });
}

int skb_pairs_detail(skb_ctx *ctx, const uint32_t *a, const uint32_t *b, int64_t n, skb_pair_detail *out) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (n < 0 || (n && (!a || !b || !out))) return fail(c, SKB_EINVAL, "bad arguments");
        if (!c->indexed || c->ix.n_indexed != c->n()) return fail(c, SKB_ESTATE, "call skb_index first");
        if (n == 0) return SKB_OK;
        std::vector<unsigned long long> hp((size_t)n);
        std::vector<int32_t> ref((size_t)n);
        for (int64_t i = 0; i < n; i++) {
            if (a[i] >= (uint32_t)c->ix.n_indexed || b[i] >= (uint32_t)c->ix.n_indexed || a[i] == b[i])
                return fail(c, SKB_EINVAL, "pair id out of range");
            hp[(size_t)i] = ((unsigned long long)a[i] << 32) | b[i];
            const uint64_t nsa = c->db.seed_off[a[i] + 1] - c->db.seed_off[a[i]], nsb = c->db.seed_off[b[i] + 1] - c->db.seed_off[b[i]];
            ref[(size_t)i] = (int32_t)(nsb < nsa ? a[i] : b[i]);
            if (!c->owns(ref[(size_t)i]))
                return fail(c, SKB_ESTATE, "the reference genome of a pair is not owned by this context (skb_set_owned)");
        }
        PoolRef<unsigned long long> d_pairs(c->pool["skb_pairs_detail.d_pairs"]);
        PoolRef<PairOut> d_out(c->pool["skb_pairs_detail.d_out"]);
        std::vector<PairOut> ho((size_t)n);
        // resident tables: every pair at once; on-demand tables: the pairs of one block of reference genomes at a time
        // resident tables: every pair at once, in input order; on-demand tables: the pairs ordered by reference genome
        // (ties in input order), one block of references -- a run of that order -- at a time
        std::vector<int64_t> order((size_t)n);
        for (int64_t i = 0; i < n; i++) order[(size_t)i] = i;
        std::vector<std::vector<int32_t>> blocks{{}};
        if (c->on_demand) {
            std::stable_sort(order.begin(), order.end(), [&](int64_t x, int64_t y) { return ref[(size_t)x] < ref[(size_t)y]; });
            std::vector<int32_t> refs;
            for (const int64_t i : order)
                if (refs.empty() || refs.back() != ref[(size_t)i]) refs.push_back(ref[(size_t)i]);
            blocks = table_blocks(c, refs);
        }
        c->blocks_last_call = c->on_demand ? (int32_t)blocks.size() : 0;
        size_t at0 = 0;
        for (const std::vector<int32_t> &blk : blocks) {
            size_t at1 = at0;  // the block's pairs: order[at0 .. at1)
            while (at1 < order.size() && (!c->on_demand || ref[(size_t)order[at1]] <= blk.back())) at1++;
            std::vector<unsigned long long> bp(at1 - at0);
            for (size_t j = 0; j < bp.size(); j++) bp[j] = hp[(size_t)order[at0 + j]];
            if (c->on_demand) build_block_tables(c, blk);
            d_pairs.upload(bp, c->st);
            d_out.reserve(bp.size(), 0, c->st);
            run_ani(c, d_pairs.p, (int64_t)bp.size(), d_out.p);
            std::vector<PairOut> bo(bp.size());
            CK(cudaMemcpyAsync(bo.data(), d_out.p, bo.size() * sizeof(PairOut), cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            for (size_t j = 0; j < bo.size(); j++) ho[(size_t)order[at0 + j]] = bo[j];
            at0 = at1;
        }
        for (int64_t i = 0; i < n; i++) {
            const PairOut &o = ho[(size_t)i];
            skb_pair_detail &d = out[i];
            d.a = a[i];
            d.b = b[i];
            d.ani = o.ani;
            d.ani_raw = o.ani_raw;
            d.af_a = o.swapped ? o.af_r : o.af_q;
            d.af_b = o.swapped ? o.af_q : o.af_r;
            d.n_anchors = o.n_anchors;
            d.n_seeds = o.n_seeds;
            d.span_q = o.span_q;
            d.span_r = o.span_r;
            d.n_chains = o.n_chains;
            d.swapped = o.swapped;
        }
        return SKB_OK;
    });
}

int skb_shared_markers(skb_ctx *ctx, const uint32_t *a, const uint32_t *b, int64_t n, int64_t *shared) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (n < 0 || (n && (!a || !b || !shared))) return fail(c, SKB_EINVAL, "bad arguments");
        if (!c->indexed || c->ix.n_indexed != c->n()) return fail(c, SKB_ESTATE, "call skb_index first");
        if (n == 0) return SKB_OK;
        for (int64_t i = 0; i < n; i++)
            if (a[i] >= (uint32_t)c->ix.n_indexed || b[i] >= (uint32_t)c->ix.n_indexed)
                return fail(c, SKB_EINVAL, "pair id out of range");
        PoolRef<uint32_t> da(c->pool["skb_shared_markers.da"]), db(c->pool["skb_shared_markers.db"]);
        PoolRef<long long> dout(c->pool["skb_shared_markers.dout"]);
        da.upload(std::vector<uint32_t>(a, a + n), c->st);
        db.upload(std::vector<uint32_t>(b, b + n), c->st);
        dout.reserve((size_t)n, 0, c->st);
        launch(c, shared_markers_kernel, nblk((uint64_t)n * 32, 256), 256, 0, c->d_markers.p, c->d_marker_off.p, da.p, db.p, n,
               dout.p);
        CK(cudaMemcpyAsync(shared, dout.p, (size_t)n * 8, cudaMemcpyDeviceToHost, c->st));
        CK(cudaStreamSynchronize(c->st));
        return SKB_OK;
    });
}

// ---- persistence: raw sketches (seeds + marker keys + host tables); the index is rebuilt on load
// v1: magic | n | n_seeds | n_marker_keys | n_contigs | tables | seeds | marker keys, sketched at m = 1000.
// v2: the same with the marker compression m (u64) between the magic and n; written only when m != 1000, so a
// default database stays a v1 file byte for byte.
static const char kMagic[8] = {'S', 'K', 'B', '2', '0', '0', 'v', '1'};
static const char kMagic2[8] = {'S', 'K', 'B', '2', '0', '0', 'v', '2'};

int skb_db_save(skb_ctx *ctx, const char *dir) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!dir) return fail(c, SKB_EINVAL, "no directory");
        const std::string path = std::string(dir) + "/sketches.skb";
        FILE *f = fopen(path.c_str(), "wb");
        if (!f) return fail(c, SKB_EIO, "cannot create " + path);
        const uint64_t n = (uint64_t)c->n(), ns = c->db.seed_off.back(), nm = c->db.n_mkeys, nc = c->db.ctg_len.size();
        std::vector<uint64_t> seeds(ns), mk(nm);
        CK(cudaStreamSynchronize(c->st));
        if (ns) CK(cudaMemcpy(seeds.data(), c->d_seeds.p, ns * 8, cudaMemcpyDeviceToHost));
        if (nm) CK(cudaMemcpy(mk.data(), c->d_mkeys.p, nm * 8, cudaMemcpyDeviceToHost));
        for (auto &s : seeds) s &= ~2ull;  // repeat flags are index state
        const bool v1 = c->marker_c == C_MARKER;
        bool ok = (v1 ? write_all(f, kMagic, 8) : write_all(f, kMagic2, 8) && write_all(f, &c->marker_c, 8)) &&
                  write_all(f, &n, 8) && write_all(f, &ns, 8) && write_all(f, &nm, 8) &&
                  write_all(f, &nc, 8) && write_all(f, c->db.seed_off.data(), (n + 1) * 8) &&
                  write_all(f, c->db.total_len.data(), n * 8) && write_all(f, c->db.ctg_off.data(), (n + 1) * 4) &&
                  write_all(f, c->db.ctg_len.data(), nc * 4) && write_all(f, seeds.data(), ns * 8) &&
                  write_all(f, mk.data(), nm * 8);
        ok = (fclose(f) == 0) && ok;
        return ok ? SKB_OK : fail(c, SKB_EIO, "short write to " + path);
    });
}

// The header and host tables of a sketches.skb (skb_db_load, skb_db_info, skb_db_load_genomes): read_db_head leaves the
// file at the seed payload, whose marker keys follow it.
struct DbHead {
    uint64_t m = C_MARKER, n = 0, ns = 0, nm = 0, nc = 0;
    std::vector<uint64_t> seed_off, total_len;
    std::vector<uint32_t> ctg_off, ctg_len;
    uint64_t digest = 1469598103934665603ull;  // FNV-1a 64 of every header and table byte, in file order
    int64_t seeds_at = 0;                      // byte offset of the seed payload
};

// "" on success, else the error
static std::string read_db_head(FILE *f, const std::string &path, DbHead &d) {
    auto rd = [&](void *p, size_t bytes) {
        if (!read_all(f, p, bytes)) return false;
        for (size_t i = 0; i < bytes; i++) d.digest = (d.digest ^ ((const unsigned char *)p)[i]) * 1099511628211ull;
        return true;
    };
    char magic[8];
    bool ok = rd(magic, 8) && (std::memcmp(magic, kMagic, 8) == 0 || (std::memcmp(magic, kMagic2, 8) == 0 && rd(&d.m, 8))) &&
              rd(&d.n, 8) && rd(&d.ns, 8) && rd(&d.nm, 8) && rd(&d.nc, 8);
    if (!ok || d.n >= GID_MASK || d.m < 1 || d.m > (uint64_t)INT64_MAX || d.nc >= (1ull << 32))
        return "not a sketch DB: " + path;
    d.seed_off.resize(d.n + 1);
    d.total_len.resize(d.n);
    d.ctg_off.resize(d.n + 1);
    d.ctg_len.resize(d.nc);
    ok = rd(d.seed_off.data(), (d.n + 1) * 8) && rd(d.total_len.data(), d.n * 8) && rd(d.ctg_off.data(), (d.n + 1) * 4) &&
         rd(d.ctg_len.data(), d.nc * 4);
    if (!ok || d.seed_off[d.n] != d.ns || d.ctg_off[d.n] != d.nc) return "truncated sketch DB: " + path;
    for (uint64_t g = 0; g < d.n; g++)
        if (d.seed_off[g] > d.seed_off[g + 1] || d.ctg_off[g] > d.ctg_off[g + 1]) return "corrupt sketch DB tables: " + path;
    d.seeds_at = (int64_t)ftello(f);
    return "";
}

int skb_db_load(skb_ctx *ctx, const char *dir) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!dir) return fail(c, SKB_EINVAL, "no directory");
        if (c->n() != 0) return fail(c, SKB_ESTATE, "context already holds genomes");
        c->genome_set++;
        const std::string path = std::string(dir) + "/sketches.skb";
        FILE *f = fopen(path.c_str(), "rb");
        if (!f) return fail(c, SKB_EIO, "cannot open " + path);
        DbHead d;
        const std::string err = read_db_head(f, path, d);
        if (!err.empty()) {
            fclose(f);
            return fail(c, SKB_EIO, err);
        }
        std::vector<uint64_t> seeds(d.ns), mk(d.nm);
        const bool ok = read_all(f, seeds.data(), d.ns * 8) && read_all(f, mk.data(), d.nm * 8);
        fclose(f);
        if (!ok) return fail(c, SKB_EIO, "truncated sketch DB: " + path);
        c->d_seeds.reserve(d.ns + 1, 0, c->st);
        c->d_mkeys.reserve(d.nm + 1, 0, c->st);
        if (d.ns) CK(cudaMemcpyAsync(c->d_seeds.p, seeds.data(), d.ns * 8, cudaMemcpyHostToDevice, c->st));
        if (d.nm) CK(cudaMemcpyAsync(c->d_mkeys.p, mk.data(), d.nm * 8, cudaMemcpyHostToDevice, c->st));
        CK(cudaStreamSynchronize(c->st));
        c->db = skb_ctx::SketchDb{std::move(d.seed_off), std::move(d.total_len), std::move(d.ctg_off), std::move(d.ctg_len),
                                  d.nm};
        c->marker_c = d.m;  // genomes added later (a search's query) are sketched at the database's density
        c->indexed = false;
        return SKB_OK;
    });
}

int skb_db_info(const char *dir, int32_t *n_genomes, int64_t *m, uint64_t *digest) {
    if (!dir) return SKB_EINVAL;
    const std::string path = std::string(dir) + "/sketches.skb";
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) return SKB_EIO;
    DbHead d;
    const bool ok = read_db_head(f, path, d).empty();
    fclose(f);
    if (!ok) return SKB_EIO;
    if (n_genomes) *n_genomes = (int32_t)d.n;
    if (m) *m = (int64_t)d.m;
    if (digest) *digest = d.digest;
    return SKB_OK;
}

// skb_db_load_genomes' marker keys.  The file's raw keys (marker << 22 | DB id) come genome by genome, ids ascending
// (skb_db_save writes what skb_add_genomes appended), so each DB genome's keys are one run [start, end).
__global__ void db_key_runs_kernel(const uint64_t *__restrict__ keys, uint64_t n, uint64_t n_db, uint32_t *__restrict__ start,
                                   uint32_t *__restrict__ end, int *__restrict__ bad) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t id = keys[i] & GID_MASK;
    const uint64_t prev = i ? keys[i - 1] & GID_MASK : ~0ull, next = i + 1 < n ? keys[i + 1] & GID_MASK : ~0ull;
    if (id >= n_db || (i && prev > id)) {  // not grouped by ascending id: the runs below would be wrong
        *bad = 1;
        return;
    }
    if (prev != id) start[id] = (uint32_t)i;
    if (next != id) end[id] = (uint32_t)(i + 1);
}
// cnt[r] = key count of the r-th requested genome (ids[r]); cnt[n] = 0 closes the scan
__global__ void db_key_counts_kernel(const int32_t *__restrict__ ids, int32_t n, const uint32_t *__restrict__ start,
                                     const uint32_t *__restrict__ end, uint32_t *__restrict__ cnt) {
    const int32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) cnt[r] = end[ids[r]] - start[ids[r]];
    if (r == n) cnt[r] = 0;
}
// Keep the keys of the requested genomes, tagged with their new ids gid0 + rank, grouped by new id ascending with each
// genome's keys in file order: a stable counting sort whose offsets `off` are the exclusive scan of the counts above.
// (retag_keys_kernel shifts every id by one constant; here the shift differs per genome.)
__global__ void db_select_keys_kernel(const uint64_t *__restrict__ keys, uint64_t n, const int32_t *__restrict__ rank,
                                      const uint32_t *__restrict__ start, const uint32_t *__restrict__ off, uint64_t gid0,
                                      uint64_t *__restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = keys[i], id = k & GID_MASK;
    const int32_t r = rank[id];
    if (r >= 0) out[off[r] + (i - start[id])] = (k & ~GID_MASK) | (gid0 + (uint64_t)r);
}

int skb_db_load_genomes(skb_ctx *ctx, const char *dir, const int32_t *ids, int32_t n) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!dir || n < 0 || (n > 0 && !ids)) return fail(c, SKB_EINVAL, "bad arguments");
        const std::string path = std::string(dir) + "/sketches.skb";
        std::unique_ptr<FILE, int (*)(FILE *)> f(fopen(path.c_str(), "rb"), fclose);
        if (!f) return fail(c, SKB_EIO, "cannot open " + path);
        DbHead d;
        const std::string err = read_db_head(f.get(), path, d);
        if (!err.empty()) return fail(c, SKB_EIO, err);
        std::vector<int32_t> rank(std::max<uint64_t>(d.n, 1), -1);  // DB id -> position in ids, -1: not requested
        uint64_t ns = 0;
        for (int32_t r = 0; r < n; r++) {
            const int32_t g = ids[r];
            if (g < 0 || (uint64_t)g >= d.n)
                return fail(c, SKB_EINVAL, "genome id " + std::to_string(g) + " out of range (" + std::to_string(d.n) + " in " + path + ")");
            if (rank[g] >= 0) return fail(c, SKB_EINVAL, "genome id " + std::to_string(g) + " requested twice");
            rank[g] = r;
            ns += d.seed_off[g + 1] - d.seed_off[g];
        }
        if (c->n() > 0 && d.m != c->marker_c)
            return fail(c, SKB_ESTATE, "the DB's marker compression " + std::to_string(d.m) + " differs from the context's " +
                                           std::to_string(c->marker_c));
        if ((uint64_t)c->n() + (uint64_t)n >= GID_MASK) return fail(c, SKB_ELIMIT, "too many genomes (22-bit ids)");
        if (d.nm >= (1ull << 32)) return fail(c, SKB_ELIMIT, "too many marker keys");
        // each genome's seeds on their own, a run of consecutive ids in one read
        std::unique_ptr<uint64_t[]> seeds(new uint64_t[ns + 1]);
        uint64_t w = 0;
        for (int32_t r = 0; r < n;) {
            int32_t r1 = r + 1;
            while (r1 < n && ids[r1] == ids[r1 - 1] + 1) r1++;
            const uint64_t a = d.seed_off[ids[r]], b = d.seed_off[ids[r1 - 1] + 1];
            if (fseeko(f.get(), d.seeds_at + (int64_t)(a * 8), SEEK_SET) != 0 || !read_all(f.get(), seeds.get() + w, (b - a) * 8))
                return fail(c, SKB_EIO, "truncated sketch DB: " + path);
            w += b - a;
            r = r1;
        }
        for (uint64_t i = 0; i < ns; i++) seeds[i] &= ~2ull;  // repeat flags are index state
        std::unique_ptr<uint64_t[]> mk(new uint64_t[d.nm + 1]);
        if (fseeko(f.get(), d.seeds_at + (int64_t)(d.ns * 8), SEEK_SET) != 0 || !read_all(f.get(), mk.get(), d.nm * 8))
            return fail(c, SKB_EIO, "truncated sketch DB: " + path);
        f.reset();

        const int32_t g0 = c->n();
        const uint64_t s0 = c->db.seed_off.back(), k0 = c->db.n_mkeys;
        if (g0 == 0) c->marker_c = d.m;  // as skb_db_load: an empty context takes the DB's m
        c->genome_set++;
        c->add_calls.push_back({g0, k0});  // skb_pop_last_add undoes it like an add
        c->d_seeds.reserve(s0 + ns + 1, s0, c->st);
        if (ns) CK(cudaMemcpyAsync(c->d_seeds.p + s0, seeds.get(), ns * 8, cudaMemcpyHostToDevice, c->st));
        uint32_t nk = 0;
        if (d.nm && n) {
            PoolRef<uint64_t> d_raw(c->pool["db_load_genomes.raw"]);
            PoolRef<int32_t> d_rank(c->pool["db_load_genomes.rank"]), d_ids(c->pool["db_load_genomes.ids"]);
            PoolRef<uint32_t> d_start(c->pool["db_load_genomes.start"]), d_end(c->pool["db_load_genomes.end"]),
                d_cnt(c->pool["db_load_genomes.cnt"]), d_off(c->pool["db_load_genomes.off"]);
            d_raw.reserve(d.nm, 0, c->st);
            CK(cudaMemcpyAsync(d_raw.p, mk.get(), d.nm * 8, cudaMemcpyHostToDevice, c->st));
            d_rank.upload(rank, c->st);
            d_ids.upload(std::vector<int32_t>(ids, ids + n), c->st);
            d_start.reserve(d.n, 0, c->st);
            d_end.reserve(d.n, 0, c->st);
            d_cnt.reserve((size_t)n + 1, 0, c->st);
            d_off.reserve((size_t)n + 1, 0, c->st);
            c->d_counter.reserve(1, 0, c->st);
            CK(cudaMemsetAsync(d_start.p, 0, d.n * 4, c->st));
            CK(cudaMemsetAsync(d_end.p, 0, d.n * 4, c->st));
            CK(cudaMemsetAsync(c->d_counter.p, 0, sizeof(int), c->st));
            launch(c, db_key_runs_kernel, nblk(d.nm, 256), 256, 0, d_raw.p, d.nm, d.n, d_start.p, d_end.p, c->d_counter.p);
            launch(c, db_key_counts_kernel, nblk((uint64_t)n + 1, 256), 256, 0, d_ids.p, n, d_start.p, d_end.p, d_cnt.p);
            exclusive_scan_u32(c, d_cnt.p, d_off.p, (size_t)n + 1);
            int bad = 0;
            CK(cudaMemcpyAsync(&nk, d_off.p + n, 4, cudaMemcpyDeviceToHost, c->st));
            CK(cudaMemcpyAsync(&bad, c->d_counter.p, sizeof(int), cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            if (bad) {
                c->add_calls.pop_back();
                return fail(c, SKB_EIO, "marker keys not grouped by ascending genome id: " + path);
            }
            c->d_mkeys.reserve(k0 + nk + 1, k0, c->st);
            launch(c, db_select_keys_kernel, nblk(d.nm, 256), 256, 0, d_raw.p, d.nm, d_rank.p, d_start.p, d_off.p,
                   (uint64_t)g0, c->d_mkeys.p + k0);
        }
        CK(cudaStreamSynchronize(c->st));
        for (int32_t r = 0; r < n; r++) {
            const int32_t g = ids[r];
            c->db.append(d.seed_off[g + 1] - d.seed_off[g], d.total_len[g], d.ctg_len.data() + d.ctg_off[g],
                         d.ctg_off[g + 1] - d.ctg_off[g]);
        }
        c->db.n_mkeys = k0 + nk;
        c->indexed = false;
        return SKB_OK;
    });
}

int skb_sketch_view_get(skb_ctx *ctx, skb_sketch_view *v) {
    if (!ctx || !v) return SKB_EINVAL;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->st);
    v->n_genomes = ctx->n();
    v->n_seeds = (int64_t)ctx->db.seed_off.back();
    v->n_marker_keys = (int64_t)ctx->db.n_mkeys;
    v->n_contigs = (int64_t)ctx->db.ctg_len.size();
    v->dev_seeds = ctx->d_seeds.p;
    v->dev_marker_keys = ctx->d_mkeys.p;
    v->host_seed_off = ctx->db.seed_off.data();
    v->host_total_len = ctx->db.total_len.data();
    v->host_ctg_off = ctx->db.ctg_off.data();
    v->host_ctg_len = ctx->db.ctg_len.data();
    return SKB_OK;
}

// ---- binary hand-off to skDER's greedy selection -------------------------------------------------------------------
// The value skDER's consumers see is the 2-decimal TEXT of an edge (`%.2f`, parsed back with stod): thresholds are
// applied to that, not to the unrounded double.  round2() reproduces it exactly: the printed hundredths
// (skb_common.cuh), one correctly rounded division.
__device__ __forceinline__ double round2(double x) { return hundredths(x) / 100.0; }
// reference src/skDER/skDERsum.cpp:107-124: an edge (col0 = a, col1 = b, ANI, AF_a, AF_b) with ANI >= min_ani gives
// genome a the member b if AF_b >= min_af, and genome b the member a if AF_a >= min_af
__global__ void summary_keys_kernel(const skb_edge *__restrict__ edges, int64_t n, double min_ani, double min_af,
                                    unsigned long long *__restrict__ keys, unsigned int *__restrict__ conn) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const skb_edge e = edges[i];
    const bool ok = round2(e.ani) >= min_ani;
    const bool a_gains = ok && round2(e.af_b) >= min_af, b_gains = ok && round2(e.af_a) >= min_af;
    keys[2 * i] = a_gains ? ((unsigned long long)e.a << 34) | ((unsigned long long)i << 1) : ~0ull;
    keys[2 * i + 1] = b_gains ? ((unsigned long long)e.b << 34) | ((unsigned long long)i << 1) | 1ull : ~0ull;
    if (a_gains) atomicAdd(&conn[e.a], 1u);
    if (b_gains) atomicAdd(&conn[e.b], 1u);
}
__global__ void summary_members_kernel(const skb_edge *__restrict__ edges, const unsigned long long *__restrict__ keys,
                                       int64_t n_keys, uint32_t *__restrict__ members) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_keys) return;
    const unsigned long long key = keys[k];
    const skb_edge &e = edges[(key & ((1ull << 34) - 1)) >> 1];
    members[k] = (key & 1ull) ? e.a : e.b;
}

__global__ void retag_keys_kernel(const uint64_t *__restrict__ in, uint64_t n, uint64_t *__restrict__ out,
                                  int64_t gid_delta) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = in[i];
    out[i] = (k & ~GID_MASK) | (uint64_t)((int64_t)(k & GID_MASK) + gid_delta);
}
__global__ void clear_rep_kernel(const uint64_t *__restrict__ in, uint64_t n, uint64_t *__restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[i] & ~2ull;
}

int skb_import_sketches(skb_ctx *ctx, int32_t n_genomes, const uint64_t *dev_seeds, int64_t n_seeds,
                        const uint64_t *dev_marker_keys, int64_t n_marker_keys, const uint64_t *host_seed_off,
                        const uint64_t *host_total_len, const uint32_t *host_ctg_off, const uint32_t *host_ctg_len,
                        int32_t keep_repeat_flags) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (n_genomes < 0 || n_seeds < 0 || n_marker_keys < 0) return fail(c, SKB_EINVAL, "bad arguments");
        if (n_genomes == 0) return SKB_OK;
        if ((uint64_t)c->n() + (uint64_t)n_genomes >= GID_MASK) return fail(c, SKB_ELIMIT, "too many genomes");
        c->genome_set++;
        const uint64_t cur = c->db.seed_off.back();
        c->add_calls.push_back({c->n(), c->db.n_mkeys});  // skb_pop_last_add undoes an import like an add
        c->d_seeds.reserve(cur + (uint64_t)n_seeds + 1, cur, c->st);
        c->d_mkeys.reserve(c->db.n_mkeys + (uint64_t)n_marker_keys + 1, c->db.n_mkeys, c->st);
        if (n_seeds && keep_repeat_flags)  // the sender indexed its genomes: their repeat flags travel with the seeds
            CK(cudaMemcpyAsync(c->d_seeds.p + cur, dev_seeds, (size_t)n_seeds * 8, cudaMemcpyDeviceToDevice, c->st));
        else if (n_seeds)
            launch(c, clear_rep_kernel, nblk((uint64_t)n_seeds, 256), 256, 0, dev_seeds, (uint64_t)n_seeds, c->d_seeds.p + cur);
        // the sender tagged its keys with ids first_src .. ; the first imported genome becomes c->n()
        if (n_marker_keys) {
            // senders export a whole context, whose ids start at 0: shift them behind this context's genomes
            launch(c, retag_keys_kernel, nblk((uint64_t)n_marker_keys, 256), 256, 0, dev_marker_keys, (uint64_t)n_marker_keys,
                   c->d_mkeys.p + c->db.n_mkeys, (int64_t)c->n());
        }
        CK(cudaStreamSynchronize(c->st));
        for (int32_t g = 0; g < n_genomes; g++)
            c->db.append(host_seed_off[g + 1] - host_seed_off[g], host_total_len[g], host_ctg_len + host_ctg_off[g],
                         host_ctg_off[g + 1] - host_ctg_off[g]);
        c->db.n_mkeys += (uint64_t)n_marker_keys;
        c->indexed = false;
        return SKB_OK;
    });
}

// Connectivity and member lists of every genome from a BINARY edge list -- what reference skDERsum
// (src/skDER/skDERsum.cpp:86-132) derives from the TSV through std::map<string, ...>: no path strings, no text parsing.
int skb_greedy_summary(skb_ctx *ctx, const skb_edge *edges, int64_t n_edges, int32_t n_genomes, double min_ani, double min_af,
                       int64_t **connectivity, int64_t **member_off, uint32_t **members) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!connectivity || !member_off || !members || n_genomes < 0) return fail(c, SKB_EINVAL, "bad arguments");
        const skb_edge *d_edges = nullptr;
        if (edges) {
            if (n_edges < 0) return fail(c, SKB_EINVAL, "bad edge count");
            for (int64_t i = 0; i < n_edges; i++)
                if (edges[i].a >= (uint32_t)n_genomes || edges[i].b >= (uint32_t)n_genomes) return fail(c, SKB_EINVAL, "edge id out of range");
            PoolRef<skb_edge> up(c->pool["greedy_summary.edges"]);
            up.reserve((size_t)std::max<int64_t>(n_edges, 1), 0, c->st);
            if (n_edges) CK(cudaMemcpyAsync(up.p, edges, (size_t)n_edges * sizeof(skb_edge), cudaMemcpyHostToDevice, c->st));
            d_edges = up.p;
        } else {  // the list the last triangle / rect left on the device
            d_edges = c->last_dev_edges;
            n_edges = c->last_n_edges;
            if (n_genomes < c->n()) return fail(c, SKB_EINVAL, "n_genomes is smaller than the context's genome count");
        }
        if (n_edges >= (1ll << 32) || n_genomes >= (1 << GID_BITS)) return fail(c, SKB_ELIMIT, "edge list too large for the summary keys");
        PoolRef<unsigned long long> d_k(c->pool["greedy_summary.keys"]), d_ks(c->pool["greedy_summary.keys_sorted"]);
        PoolRef<unsigned int> d_conn(c->pool["greedy_summary.conn"]);
        PoolRef<uint32_t> d_mem(c->pool["greedy_summary.members"]);
        const size_t nk = 2 * (size_t)n_edges;
        d_k.reserve(std::max<size_t>(nk, 1), 0, c->st);
        d_ks.reserve(std::max<size_t>(nk, 1), 0, c->st);
        d_conn.reserve((size_t)n_genomes + 1, 0, c->st);
        d_mem.reserve(std::max<size_t>(nk, 1), 0, c->st);
        CK(cudaMemsetAsync(d_conn.p, 0, ((size_t)n_genomes + 1) * 4, c->st));
        std::vector<unsigned int> h_conn((size_t)n_genomes);
        if (n_edges) {
            launch(c, summary_keys_kernel, nblk((uint64_t)n_edges, 256), 256, 0, d_edges, n_edges, min_ani, min_af, d_k.p, d_conn.p);
            sort_keys_u64(c, (const uint64_t *)d_k.p, (uint64_t *)d_ks.p, nk, 56);  // unused keys (all ones) sort last
        }
        if (n_genomes) CK(cudaMemcpyAsync(h_conn.data(), d_conn.p, (size_t)n_genomes * 4, cudaMemcpyDeviceToHost, c->st));
        CK(cudaStreamSynchronize(c->st));
        int64_t *conn = (int64_t *)std::malloc(sizeof(int64_t) * (size_t)std::max(n_genomes, 1));
        int64_t *off = (int64_t *)std::malloc(sizeof(int64_t) * ((size_t)n_genomes + 1));
        if (!conn || !off) {
            std::free(conn);
            std::free(off);
            return fail(c, SKB_ENOMEM, "host out of memory");
        }
        off[0] = 0;
        for (int32_t g = 0; g < n_genomes; g++) {
            conn[g] = h_conn[(size_t)g];
            off[g + 1] = off[g] + conn[g];
        }
        const int64_t total = off[n_genomes];
        uint32_t *mem = (uint32_t *)std::malloc(sizeof(uint32_t) * (size_t)std::max<int64_t>(total, 1));
        if (!mem) {
            std::free(conn);
            std::free(off);
            return fail(c, SKB_ENOMEM, "host out of memory");
        }
        if (total) {
            launch(c, summary_members_kernel, nblk((uint64_t)total, 256), 256, 0, d_edges, d_ks.p, total, d_mem.p);
            CK(cudaMemcpyAsync(mem, d_mem.p, (size_t)total * 4, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
        }
        *connectivity = conn;
        *member_off = off;
        *members = mem;
        return SKB_OK;
    });
}

// ---- skani's triangle --full-matrix [--distance] (skb_matrix.cuh) ---------------------------------------------------
int skb_write_matrix(skb_ctx *ctx, const char *path, int32_t kind, const skb_edge *edges, int64_t n_edges,
                     int32_t n_genomes, const char *labels, const int64_t *label_off) {
    return guarded(ctx, [&]() -> int {
        skb_ctx *c = ctx;
        if (!path || n_genomes < 0 || !label_off) return fail(c, SKB_EINVAL, "bad arguments");
        if (kind != SKB_MATRIX_ANI && kind != SKB_MATRIX_DISTANCE && kind != SKB_MATRIX_AF)
            return fail(c, SKB_EINVAL, "unknown matrix kind " + std::to_string(kind));
        const int32_t n = n_genomes;
        if (label_off[0] != 0) return fail(c, SKB_EINVAL, "label offsets must start at 0");
        int64_t max_label = 0;
        for (int32_t g = 0; g < n; g++) {
            if (label_off[g + 1] < label_off[g]) return fail(c, SKB_EINVAL, "label offsets must not decrease");
            max_label = std::max(max_label, label_off[g + 1] - label_off[g]);
        }
        if (label_off[n] && !labels) return fail(c, SKB_EINVAL, "no label bytes");
        const skb_edge *d_edges = nullptr;
        if (edges) {
            if (n_edges < 0) return fail(c, SKB_EINVAL, "bad edge count");
            for (int64_t i = 0; i < n_edges; i++) {
                const skb_edge &e = edges[i];
                if (!(e.a < e.b && e.b < (uint32_t)n)) return fail(c, SKB_EINVAL, "edge " + std::to_string(i) + ": ids out of range");
                if (i && !(edges[i - 1].a < e.a || (edges[i - 1].a == e.a && edges[i - 1].b < e.b)))
                    return fail(c, SKB_EINVAL, "edge " + std::to_string(i) + ": the list is not strictly increasing in (a, b)");
                for (double x : {e.ani, e.af_a, e.af_b})
                    if (!(x >= 0.0 && x <= 100.0)) return fail(c, SKB_EINVAL, "edge " + std::to_string(i) + ": a value outside [0, 100]");
            }
            if (n_edges >= (1ll << 31)) return fail(c, SKB_ELIMIT, "too many edges for the 32-bit cell map");
            PoolRef<skb_edge> up(c->pool["matrix.edges"]);
            up.reserve((size_t)std::max<int64_t>(n_edges, 1), 0, c->st);
            if (n_edges) CK(cudaMemcpyAsync(up.p, edges, (size_t)n_edges * sizeof(skb_edge), cudaMemcpyHostToDevice, c->st));
            d_edges = up.p;
        } else {
            if (c->whole_triangle < 0 || (uint64_t)c->whole_triangle != c->genome_set)
                return fail(c, SKB_ESTATE, "no whole-triangle edge list: the last edge call was not a whole skb_triangle, or "
                                           "genomes were added, removed or cleared since");
            if (n != c->n()) return fail(c, SKB_EINVAL, "n_genomes differs from the context's genome count");
            d_edges = c->last_dev_edges;
            n_edges = c->last_n_edges;
            if (n_edges >= (1ll << 31)) return fail(c, SKB_ELIMIT, "too many edges for the 32-bit cell map");
        }
        // rows per block: the cell map (4 bytes a cell), the row offsets and the text (at most 7 bytes a cell of values
        // in [0, 100]) of R rows within the budget and within what the device has free
        const char *mb = std::getenv("SKB_MATRIX_BLOCK_MB");
        const uint64_t budget = (uint64_t)(mb && std::atoll(mb) > 0 ? std::atoll(mb) : 1024) << 20;
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        const uint64_t per_row = 4ull * (uint64_t)n + 16 + (uint64_t)max_label + 1 + 7ull * (uint64_t)n;
        const uint64_t room = free_b / 10 * 9;
        if (n && per_row > room) return fail(c, SKB_ELIMIT, "one matrix row does not fit the device");
        const int32_t R = n ? (int32_t)std::clamp<uint64_t>(std::min(budget, room) / per_row, 1, (uint64_t)n) : 0;

        struct File {
            FILE *f;
            ~File() { if (f) fclose(f); }
        } out{fopen(path, "wb")};
        if (!out.f) return fail(c, SKB_EIO, std::string("cannot create ") + path);
        const std::string first = std::to_string(n) + "\n";
        if (!write_all(out.f, first.data(), first.size())) return fail(c, SKB_EIO, std::string("write failed: ") + path);
        if (n == 0) {
            FILE *f = out.f;
            out.f = nullptr;
            return fclose(f) == 0 ? SKB_OK : fail(c, SKB_EIO, std::string("write failed: ") + path);
        }
        PoolRef<char> d_labels(c->pool["matrix.labels"]), d_text(c->pool["matrix.text"]);
        PoolRef<int64_t> d_label_off(c->pool["matrix.label_off"]);
        PoolRef<int32_t> d_map(c->pool["matrix.map"]);
        PoolRef<uint64_t> d_len(c->pool["matrix.row_len"]), d_off(c->pool["matrix.row_off"]);
        d_labels.reserve((size_t)label_off[n] + 1, 0, c->st);
        if (label_off[n]) CK(cudaMemcpyAsync(d_labels.p, labels, (size_t)label_off[n], cudaMemcpyHostToDevice, c->st));
        d_label_off.reserve((size_t)n + 1, 0, c->st);
        CK(cudaMemcpyAsync(d_label_off.p, label_off, ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, c->st));
        d_map.reserve((size_t)R * n, 0, c->st);
        d_len.reserve((size_t)R + 1, 0, c->st);
        d_off.reserve((size_t)R + 1, 0, c->st);
        d_text.reserve((size_t)R * (per_row - 4ull * n - 16), 0, c->st);

        struct Events {
            cudaEvent_t rendered = nullptr, copied[2] = {};
            ~Events() {
                for (cudaEvent_t e : {rendered, copied[0], copied[1]})
                    if (e) cudaEventDestroy(e);
            }
        } ev;
        if (!c->st_copy) CK(cudaStreamCreateWithFlags(&c->st_copy, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ev.rendered, cudaEventDisableTiming));
        for (cudaEvent_t &e : ev.copied) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        // block k: the map, the row lengths and their scan, the block's size to the host; then its text is written on
        // st and copied into pinned slot k % 2 on st_copy while the host writes block k - 1 to the file
        uint64_t bytes[2] = {0, 0};
        int64_t k = 0;
        struct Drain {  // whatever else happens, no copy into a pinned slot is in flight when the call returns
            cudaStream_t s;
            ~Drain() { cudaStreamSynchronize(s); }
        } drain{c->st_copy};
        for (int32_t r0 = 0; r0 < n; r0 += R, k++) {
            const int32_t rows = std::min(R, n - r0);
            const int s = (int)(k & 1);
            CK(cudaMemsetAsync(d_map.p, 0xff, (size_t)rows * n * 4, c->st));
            if (n_edges)
                launch(c, matrix_scatter_kernel, nblk((uint64_t)n_edges, 256), 256, 0, d_edges, n_edges, n, r0, rows, d_map.p);
            launch(c, matrix_row_len_kernel, (unsigned)rows, MX_THREADS, 0, d_map.p, d_edges, d_label_off.p, n, r0, kind, d_len.p);
            CK(cudaMemsetAsync(d_len.p + rows, 0, 8, c->st));
            cub_run(c, 2, [&](void *tmp, size_t &b) {
                return cub::DeviceScan::ExclusiveSum(tmp, b, d_len.p, d_off.p, rows + 1, c->st);
            });
            CK(cudaMemcpyAsync(&bytes[s], d_off.p + rows, 8, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            if (bytes[s] > d_text.b.cap) {  // values outside [0, 100] print longer: the previous copy must be done
                if (k) CK(cudaEventSynchronize(ev.copied[s ^ 1]));
                d_text.reserve(bytes[s], 0, c->st);
            }
            if (bytes[s] > c->h_matrix_cap[s]) {  // slot s last held block k - 2, written to the file already
                if (c->h_matrix[s]) CK(cudaFreeHost(c->h_matrix[s]));
                c->h_matrix[s] = nullptr;
                c->h_matrix_cap[s] = 0;
                CK(cudaHostAlloc((void **)&c->h_matrix[s], bytes[s], cudaHostAllocDefault));
                c->h_matrix_cap[s] = bytes[s];
            }
            if (k) CK(cudaStreamWaitEvent(c->st, ev.copied[s ^ 1], 0));  // d_text is free once block k - 1 is copied out
            launch(c, matrix_write_kernel, (unsigned)rows, MX_THREADS, 0, d_map.p, d_edges, d_labels.p, d_label_off.p, n, r0,
                   kind, d_off.p, d_text.p);
            CK(cudaEventRecord(ev.rendered, c->st));
            CK(cudaStreamWaitEvent(c->st_copy, ev.rendered, 0));
            CK(cudaMemcpyAsync(c->h_matrix[s], d_text.p, bytes[s], cudaMemcpyDeviceToHost, c->st_copy));
            CK(cudaEventRecord(ev.copied[s], c->st_copy));
            if (k) {
                CK(cudaEventSynchronize(ev.copied[s ^ 1]));
                if (!write_all(out.f, c->h_matrix[s ^ 1], bytes[s ^ 1])) return fail(c, SKB_EIO, std::string("write failed: ") + path);
            }
        }
        const int s = (int)((k - 1) & 1);
        CK(cudaEventSynchronize(ev.copied[s]));
        if (!write_all(out.f, c->h_matrix[s], bytes[s])) return fail(c, SKB_EIO, std::string("write failed: ") + path);
        FILE *f = out.f;
        out.f = nullptr;
        return fclose(f) == 0 ? SKB_OK : fail(c, SKB_EIO, std::string("write failed: ") + path);
    });
}

}  // extern "C"
