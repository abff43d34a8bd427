/*
 * skani_b200.h -- C-ABI of the B200-native all-vs-all ANI/AF engine (libskani_b200.so).
 *
 * The reference (raufs/skDER) has no FFI for this path: its boundary is `argv + files` to the
 * external `skani` program (reference src/skDER/util.py:636-652 runCmd; call sites
 * src/skDER/skder.py:16-18 triangle, :58-59 dist, :103 sketch, :119 search;
 * src/skDER/cidder.py:362-363 dist).  Each entry point below names the skani sub-command /
 * call site it stands in for.  The `skani` command-line shim (skder_b200/cli.py) maps argv onto
 * these calls; INTEGRATION.md shows the ctypes stub a skDER maintainer would add instead.
 *
 * Conventions: every function returns 0 on success, a negative SKB_E* code otherwise (never
 * throws, never falls back to a CPU path); skb_last_error() gives the message.  Buffers passed in
 * are caller-owned HOST memory unless the name says `dev`.  Buffers returned through `**out` are
 * library-owned and released with skb_free().
 */
#ifndef SKANI_B200_H
#define SKANI_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SKB_OK 0
#define SKB_EINVAL (-1)
#define SKB_ECUDA (-2)
#define SKB_EIO (-3)
#define SKB_ENOMEM (-4)
#define SKB_ESTATE (-5)
#define SKB_ELIMIT (-6)

typedef struct skb_ctx skb_ctx;

/* ---- parameters of the estimator (defaults = skani defaults as restated in DESIGN.md) ------- */
typedef struct {
    int32_t min_contig_len; /* 500  */
    int32_t chunk_len;      /* 20000 */
    int32_t band_bp;        /* 2500 */
    int32_t max_gap;        /* 300 */
    int32_t anchor_score;   /* 20 */
    int32_t min_anchors;    /* 3 */
    int32_t min_score;      /* 45 */
    int32_t max_mult;       /* 8 */
    int32_t max_chunk_chains; /* 8 */
    int32_t ovl_num, ovl_den; /* 1/2 */
    int32_t span_ext;       /* 170 */
    double debias_a, debias_g; /* learned-debias substitute: 100-ANI = a*(100-raw)^g */
} skb_params;
void skb_default_params(skb_params *p);

/* ---- host-side FASTA ingest + 2-bit packing (skani's file reader; invoked for every path in
 *      the `-l` / `--rl` / `--ql` list files and for `skani search <fasta>`) ------------------- */
typedef struct {
    uint64_t *words;      /* 2-bit codes, 32 bases / word, base j at bits 2*(j%32); kept contigs concatenated */
    int64_t n_words;      /* even (16-byte multiple) */
    int64_t n_bases;      /* sum of kept contig lengths */
    int32_t n_contigs;    /* kept contigs */
    int64_t *contig_lens; /* [n_contigs] */
    char *first_name;     /* header line of first kept record, without '>' */
    int64_t n50;          /* N50 over ALL records (reference src/skDER/util.py:686-724 n50_calc) */
    int64_t total_bases_all; /* over all records */
    char **contig_names;  /* [n_contigs] header lines of the kept records, without '>' (skb_pack_contigs: NULL) */
} skb_packed;
int skb_pack_fasta(const char *path, int32_t min_contig_len, skb_packed **out);
/* n files on n_threads host threads; out[i] is NULL where file i failed (return value = #failures) */
int skb_pack_fasta_many(const char *const *paths, int32_t n, int32_t min_contig_len, int32_t n_threads,
                        skb_packed **out);
/* from ASCII contigs already in memory (tests, synthetic benches) */
int skb_pack_contigs(const char *const *seqs, const int64_t *lens, int32_t n, int32_t min_contig_len,
                     skb_packed **out);
void skb_packed_free(skb_packed *p);

/* ---- context ------------------------------------------------------------------------------- */
int skb_create(int32_t device, const skb_params *params, skb_ctx **out);
void skb_destroy(skb_ctx *ctx);
const char *skb_last_error(const skb_ctx *ctx); /* ctx may be NULL: last creation error */

/* ---- sketching: `skani sketch -l list -o db` (skder.py:103) and the sketch phase of
 *      `skani triangle` / `skani dist` ------------------------------------------------------- */
/* Upload n packed genomes (host pointers, pinned or pageable), sketch them on the device and
 * append them to the context's sketch DB.  Genome ids are assigned in call order. */
int skb_add_genomes(skb_ctx *ctx, int32_t n, const skb_packed *const *genomes);
/* skani's per-sequence mode (-i, --qi, --ri; DESIGN.md section 3): every kept contig of every one of the n_files packed
 * files becomes a genome of its own with one contig, ids in (file, record) order -- its sketch is exactly the one the
 * record gets as a one-contig genome of skb_add_genomes.  Uploads and batches as skb_add_genomes; one skb_pop_last_add
 * undoes the whole call.  SKB_ELIMIT: more genomes than 22-bit ids, a record too large for 31-bit padded coordinates,
 * or a file of 2^32 bases or more. */
int skb_add_sequences(skb_ctx *ctx, int32_t n_files, const skb_packed *const *files);
/* Build the search structures (inverted marker index, per-genome seed hash indices, chunk tables)
 * over every genome added so far.  Must be called before triangle/rect; may be called again after
 * more genomes were added. */
int skb_index(skb_ctx *ctx);
/* Index the genomes added since the last skb_index / skb_index_append as QUERY-ONLY additions (seed
 * tables, chunk tables, marker lists appended; inverted index untouched): they may be queries of skb_rect,
 * not references and not part of a triangle.  With skb_pop_last_add this is `skani search` (skder.py:119)
 * against a resident database: one query genome comes and goes at the cost of its own sketch. */
int skb_index_append(skb_ctx *ctx);
/* Undo the most recent skb_add_genomes / skb_add_sequences call (only genomes that are not in the inverted index). */
int skb_pop_last_add(skb_ctx *ctx);
int32_t skb_n_genomes(const skb_ctx *ctx);
/* drop every genome and index but keep the device allocations (repeated runs on one context) */
int skb_clear(skb_ctx *ctx);

/* sketch read-back (parity tests; DB persistence) */
int skb_sketch_sizes(skb_ctx *ctx, int32_t g, int64_t *n_seeds, int64_t *n_markers, int32_t *n_chunks,
                     int64_t *total_len);
int skb_get_seeds(skb_ctx *ctx, int32_t g, uint64_t *out);   /* position-ordered packed seed records */
int skb_get_markers(skb_ctx *ctx, int32_t g, uint64_t *out); /* sorted unique canonical 21-mers */

/* skani's -m (DESIGN.md section 3): a canonical 21-mer is a marker iff its hash is below UINT64_MAX / m (integer
 * division; default m = 1000).  Markers only decide which pairs the prescreen passes; seeds, chains and the ANI/AF of a
 * pair are the same at every m.  Context state, kept across skb_clear, applied to every later skb_add_genomes.  m < 1:
 * SKB_EINVAL; a different m while the context holds genomes: SKB_ESTATE (setting the current value is fine).  A small
 * m makes many markers: like any other allocation, one the device cannot hold fails the call that needs it. */
int skb_set_marker_compression(skb_ctx *ctx, int64_t m);
int skb_marker_compression(const skb_ctx *ctx, int64_t *m);

/* persistence of the sketch DB: `skani sketch -o <dir>` writes it, `skani search -d <dir>` loads it.  The file records
 * the marker compression (format SKB200v1 at m = 1000, SKB200v2 otherwise); skb_db_load reads both and sets the
 * context's m to the file's, so genomes added afterwards (a search's query) are sketched at the database's density. */
int skb_db_save(skb_ctx *ctx, const char *dir);
int skb_db_load(skb_ctx *ctx, const char *dir);
/* What dir/sketches.skb holds, read from its header and host tables only (no seed or marker payload, no context, no
 * device): its genome count, its marker compression m, and a 64-bit digest (FNV-1a) of every header and table byte --
 * which changes whenever the file is rewritten with other genomes.  SKB_EIO for a missing or malformed file. */
int skb_db_info(const char *dir, int32_t *n_genomes, int64_t *m, uint64_t *digest);
/* Append the DB genomes ids[0 .. n) of dir/sketches.skb to the context, in that order, as one skb_add_genomes of the same
 * FASTAs would: genome ids[r] becomes id n_before + r, with the seeds (repeat flags clear), contig tables and marker keys
 * the add would have made, so seeds, markers and every edge are bit-identical.  Each genome's seeds are read from the
 * file on their own; the marker keys are selected, re-tagged and grouped by the new id on the device.  Works on an empty
 * or non-empty context before skb_index; one skb_pop_last_add undoes it.  An empty context takes the file's m (as
 * skb_db_load); a non-empty one with another m: SKB_ESTATE.  An id out of range or repeated: SKB_EINVAL.  A missing or
 * malformed file: SKB_EIO. */
int skb_db_load_genomes(skb_ctx *ctx, const char *dir, const int32_t *ids, int32_t n);

/* ---- pair results --------------------------------------------------------------------------- */
typedef struct {
    uint32_t a, b;  /* genome ids; for triangle a < b */
    double ani;     /* percent, unrounded */
    double af_a;    /* percent aligned fraction of genome a */
    double af_b;
} skb_edge;

typedef struct {
    uint32_t a, b;
    double ani, ani_raw, af_a, af_b; /* fractions in [0,1]; ani < 0 if no estimate */
    int64_t n_anchors, n_seeds, span_q, span_r;
    int32_t n_chains, swapped;
} skb_pair_detail;

typedef struct {
    int64_t n_pairs_total;    /* pairs in scope of this call (this partition) */
    int64_t n_pairs_screened; /* pairs that passed the marker prescreen */
    int64_t n_edges;
    float ms_screen, ms_ani, ms_total; /* device time (CUDA events) */
    int64_t launches;         /* kernels launched by this call */
    int64_t sum_query_seeds;  /* sum over screened pairs of the query genome's seed count (roofline bytes) */
    int64_t sum_anchors;      /* sum over screened pairs of chained anchors (roofline bytes) */
    float ms_anchor;          /* device time of the anchor kernel (dominant kernel), summed over its launches */
    int32_t n_anchor_launches;
} skb_stats;

/* `skani triangle -l list --min-af A -E -s S` (skder.py:16-18): all pairs a<b of the DB whose
 * row a belongs to partition `part` of `n_parts` (rows are dealt in zig-zag order 0..P-1,P-1..0,... so that all partitions
 * hold the same number of pairs; use 0,1 for the whole triangle).  screen_pct = skani -s (percent; <=0 disables), min_af_pct = skani --min-af. */
int skb_triangle(skb_ctx *ctx, double screen_pct, double min_af_pct, int32_t part, int32_t n_parts,
                 skb_edge **edges, int64_t *n_edges, skb_stats *stats);

/* `skani dist --rl R --ql Q` (skder.py:58-59, cidder.py:362-363) and `skani search q -d db`
 * (skder.py:119): every (ref, query) pair of the two id lists.  In each edge a = ref id, b = query id. */
int skb_rect(skb_ctx *ctx, const int32_t *refs, int32_t n_refs, const int32_t *queries, int32_t n_queries,
             double screen_pct, double min_af_pct, skb_edge **edges, int64_t *n_edges, skb_stats *stats);

/* skani's -n on dist / search (DESIGN.md section 3): every later skb_rect keeps, for each query genome, only its first n
 * edges in row order -- ANI descending (the unrounded double), ties to the lower reference id -- after the screen,
 * --min-af and the active estimator.  The kept edges stay in skb_rect's (a, b) order, and skb_device_edges,
 * skb_last_edge_ci, skb_last_edge_detail and skb_greedy_summary(edges = NULL) see only them.  n = 0 (the default): all
 * edges.  Context state, kept across skb_clear.  skb_triangle and skb_pairs_edges are unaffected: skani's triangle has
 * no -n.  n < 0: SKB_EINVAL. */
int skb_set_max_results(skb_ctx *ctx, int64_t n);

/* How a pair's accepted chains become one ANI (skani's default, --median, --robust; DESIGN.md section 3).  Context
 * state, kept across skb_clear: applies to every later skb_triangle, skb_rect, skb_pairs_edges and skb_pairs_detail
 * call.  AF, chain, anchor and seed counts are the same in every mode.  Any other value: SKB_EINVAL. */
#define SKB_ANI_MEAN 0
#define SKB_ANI_MEDIAN 1
#define SKB_ANI_ROBUST 2
int skb_set_ani_estimator(skb_ctx *ctx, int32_t estimator);

/* skani's --ci (DESIGN.md section 3): a percentile-bootstrap interval of every edge's ANI (100 replicates of the pair's
 * accepted chains; 5th and 95th percentile).  Context state, kept across skb_clear: enabled != 0 applies to every later
 * skb_triangle, skb_rect and skb_pairs_edges call, which return SKB_EINVAL while it is on and the estimator is not
 * SKB_ANI_MEAN.  The edges themselves are the same with and without it. */
int skb_set_ani_ci(skb_ctx *ctx, int32_t enabled);
/* The intervals of the edge list of the last skb_triangle, skb_rect or skb_pairs_edges call on this context (also one
 * made with edges == NULL), in edge order: lo_hi[2 i] and lo_hi[2 i + 1] are edge i's lower and upper bound, percent on
 * the ANI's scale, copied from the per-edge records skb_last_edge_detail serves (ani_lo, ani_hi); *n = that call's
 * edge count.  malloc'ed (skb_free).  SKB_ESTATE if that call ran without --ci, also when it ran with --detailed. */
int skb_last_edge_ci(skb_ctx *ctx, double **lo_hi, int64_t *n);

/* skani's --detailed (DESIGN.md section 3): per edge, what the extra columns need beyond the contig statistics below.
 * "a" / "b" are the edge's genomes (skb_edge.a / .b). */
typedef struct {
    double ani_lo, ani_hi;          /* percent: the --ci interval; skb_last_edge_ci reads it from here */
    double sd;                      /* percent: seed-weighted standard deviation of the accepted chains' ANI */
    int64_t covered_a, covered_b;   /* bases of genome a / b in the accepted chains' extended spans (AF numerators) */
    int32_t n_chains, pad;          /* accepted chains */
} skb_edge_detail;                  /* 48 bytes */
/* Context state, kept across skb_clear: enabled != 0 applies to every later skb_triangle, skb_rect and skb_pairs_edges
 * call, which return SKB_EINVAL while it is on and the estimator is not SKB_ANI_MEAN.  The edges themselves are the same
 * with and without it. */
int skb_set_detailed(skb_ctx *ctx, int32_t enabled);
/* The details of the edge list of the last skb_triangle, skb_rect or skb_pairs_edges call on this context (also one
 * made with edges == NULL), in edge order; *n = that call's edge count.  malloc'ed (skb_free).  SKB_ESTATE if that call
 * ran without --detailed, also when it ran with --ci. */
int skb_last_edge_detail(skb_ctx *ctx, skb_edge_detail **out, int64_t *n);
/* Host-side statistics of the kept contigs (those of at least min_contig_len: what the sketch DB holds) of genomes
 * first .. first + n - 1: n_contigs[i], and nx[3 i .. 3 i + 2] = N90, N50, N10 (DESIGN.md section 3; 0 for a genome
 * without kept contigs).  Serves added, loaded and imported genomes alike. */
int skb_genome_contig_stats(skb_ctx *ctx, int32_t first, int32_t n, int32_t *n_contigs, int64_t *nx);

/* explicit pair list, full detail, no screening / no AF filter (parity tests) */
int skb_pairs_detail(skb_ctx *ctx, const uint32_t *a, const uint32_t *b, int64_t n, skb_pair_detail *out);
/* shared-marker counts of an explicit pair list (prescreen parity) */
int skb_shared_markers(skb_ctx *ctx, const uint32_t *a, const uint32_t *b, int64_t n, int64_t *shared);

/* ---- device-resident sketch exchange (multi-GPU replication over NCCL; the host side wraps these
 *      pointers as torch tensors) ------------------------------------------------------------- */
typedef struct {
    int32_t n_genomes;
    int64_t n_seeds, n_marker_keys, n_contigs;
    uint64_t *dev_seeds;        /* [n_seeds] */
    uint64_t *dev_marker_keys;  /* [n_marker_keys] (marker << 22 | genome id), unsorted */
    uint64_t *host_seed_off;    /* [n_genomes+1] */
    uint64_t *host_total_len;   /* [n_genomes] */
    uint32_t *host_ctg_off;     /* [n_genomes+1] */
    uint32_t *host_ctg_len;     /* [n_contigs] */
} skb_sketch_view;
int skb_sketch_view_get(skb_ctx *ctx, skb_sketch_view *view);
/* append genomes whose sketches were produced by another context (device pointers on THIS device);
 * marker keys are re-tagged with the receiving context's genome ids.  The sender's marker compression is not part of
 * the view: the caller must give both contexts the same one (skb_set_marker_compression; multi.py checks it). */
int skb_import_sketches(skb_ctx *ctx, int32_t n_genomes, const uint64_t *dev_seeds, int64_t n_seeds,
                        const uint64_t *dev_marker_keys, int64_t n_marker_keys, const uint64_t *host_seed_off,
                        const uint64_t *host_total_len, const uint32_t *host_ctg_off, const uint32_t *host_ctg_len,
                        int32_t keep_repeat_flags /* 1: the sender ran skb_index, its repeat flags travel with the seeds */);

/* ---- the triangle on several GPUs, sharded by REFERENCE genome (skder_b200/multi.py; SURVEY.md section 8e) ----------
 * Every context holds all sketches (replicated) but builds seed tables only for the genomes it owns, a contiguous id
 * range set before skb_index.  The triangle then runs in two steps with one small exchange in between: each rank
 * screens its rows (skb_screen_triangle leaves the surviving pairs on the device), the pair lists are all-gathered,
 * and each rank evaluates the pairs whose reference genome -- the one with more seeds -- it owns (skb_pairs_edges with
 * owned_only).  Every rank therefore probes only tables it built itself, and a reference's pairs stay together on one
 * GPU (L2 reuse), however the survivors are distributed over the rows. */
int skb_set_owned(skb_ctx *ctx, int32_t first, int32_t count); /* count = -1: all genomes (the default) */
/* A rank builds the seed tables and repeat flags of its OWN genomes before the exchange (skb_index_seed_tables: the first
 * half of skb_index), keeps them across the reset (skb_clear_keep_tables instead of skb_clear), imports everybody's
 * sketches with their repeat flags, declares the same genomes owned, and calls skb_index: the tables are reused, only the
 * chunk tables and the marker index of the whole set are built.  Table work and memory per rank: 1/P, done once. */
int skb_index_seed_tables(skb_ctx *ctx);
int skb_clear_keep_tables(skb_ctx *ctx);
int skb_screen_triangle(skb_ctx *ctx, double screen_pct, int32_t part, int32_t n_parts, const uint64_t **dev_pairs,
                        int64_t *n_pairs, skb_stats *stats);
/* dev_pairs: (a << 32 | b) on this device; edges may be NULL (result stays on the device, skb_device_edges) */
int skb_pairs_edges(skb_ctx *ctx, const uint64_t *dev_pairs, int64_t n_pairs, int32_t owned_only, double min_af_pct,
                    skb_edge **edges, int64_t *n_edges, skb_stats *stats);

/* Device copy of the edge list produced by the last skb_triangle / skb_rect call on this context (same order
 * as the host copy; valid until the next call on the context).  skb_triangle accepts edges == NULL: the result
 * then stays on the device only -- what a multi-GPU caller wants, which gathers the per-rank lists over NCCL
 * (skder_b200/multi.py) instead of bouncing them through host memory. */
int skb_device_edges(skb_ctx *ctx, const skb_edge **dev_edges, int64_t *n_edges);

/* ---- binary edge hand-off to skDER's greedy selection (SURVEY.md section 8 f3) --------------------------------------
 * What reference skDERsum (src/skDER/skDERsum.cpp:86-132) computes from the edge TSV: per genome, how many genomes it
 * covers (connectivity) and which (members, in edge order).  An edge (a, b, ANI, AF_a, AF_b) whose printed ANI is >=
 * min_ani gives a the member b if the printed AF_b >= min_af, and b the member a if the printed AF_a >= min_af
 * (skDERsum.cpp:112-124); "printed" = the 2-decimal text skani writes, reproduced exactly on the device.
 * edges: host array, or NULL for the list the last skb_triangle / skb_rect call left on the device.  Results are
 * malloc'ed (skb_free): connectivity[n_genomes], member_off[n_genomes + 1], members[member_off[n_genomes]].
 * The host side (skder_b200/select.py) multiplies by N50 and writes Genome_Information_for_Greedy_Clustering.txt
 * byte-identical to the reference helper's. */
int skb_greedy_summary(skb_ctx *ctx, const skb_edge *edges, int64_t n_edges, int32_t n_genomes, double min_ani, double min_af,
                       int64_t **connectivity, int64_t **member_off, uint32_t **members);

/* ---- skani's `triangle --full-matrix [--distance]` (DESIGN.md section 3) -------------------------------------------
 * Writes the whole file at `path`: the line "N\n" (N = n_genomes), then per genome r in id order its label (labels
 * bytes label_off[r] .. label_off[r + 1]), for every genome c in id order '\t' and the cell (r, c) as `%.2f` text, then
 * '\n'.  The value of a cell is read from the edge {r, c}'s printed `%.2f` text, in hundredths:
 *   SKB_MATRIX_ANI       r = c: 100.00; an edge: its ANI; no edge: 0.00.
 *   SKB_MATRIX_DISTANCE  100.00 minus the SKB_MATRIX_ANI cell, computed on the printed hundredths (10000 - cents), so
 *                        the two files are exact complements: the diagonal 0.00, no edge 100.00.
 *   SKB_MATRIX_AF        r = c: 100.00; an edge: genome r's aligned fraction (af_a if r is the edge's a, else af_b), so
 *                        the matrix is not symmetric; no edge: 0.00.
 * edges == NULL: the device edge list of the last skb_triangle (the one skb_device_edges serves); n_edges is ignored and
 * n_genomes must equal the context's genome count.  SKB_ESTATE if the last edge call was skb_rect or skb_pairs_edges,
 * a partition of the triangle (n_parts > 1), or if genomes were added, removed or cleared since.
 * edges != NULL: a host list, strictly increasing in (a, b), a < b < n_genomes, every value finite in [0, 100];
 * otherwise SKB_EINVAL.  A multi-GPU rank holding a gathered list passes it this way.
 * The text is rendered on the device in blocks of rows (at most SKB_MATRIX_BLOCK_MB MiB of device scratch, default
 * 1024) and written while the next block renders.  SKB_EINVAL for an unknown kind, SKB_EIO on a write failure (the file
 * may then be partial: the caller makes the write atomic), SKB_ELIMIT if one row does not fit the device. */
#define SKB_MATRIX_ANI 0
#define SKB_MATRIX_DISTANCE 1
#define SKB_MATRIX_AF 2
int skb_write_matrix(skb_ctx *ctx, const char *path, int32_t kind, const skb_edge *edges, int64_t n_edges,
                     int32_t n_genomes, const char *labels, const int64_t *label_off /* [n_genomes + 1] */);

void skb_free(void *p);

/* Seed tables of the genomes a pair compares against (DESIGN.md section 2).  skb_index keeps every genome's table resident
 * when they fit the table budget -- the density's budget of device memory, but at least half of the memory free, capped
 * by SKB_TABLE_BUDGET_MB (MiB) -- and otherwise switches the context to on-demand tables: every edge call (skb_triangle,
 * skb_rect, skb_pairs_edges, skb_pairs_detail) then builds the tables of the genomes that are the reference of a
 * surviving pair, in blocks that fit the budget, and merges the blocks' results by each pair's position in the call's
 * pair list, into the order one resident pass leaves; every result is the same.  A context with skb_set_owned keeps its
 * tables resident.  *on_demand: 1 if the last skb_index chose on-demand tables; *blocks_last_call: the blocks the last
 * edge call built (0 with resident tables).  Either pointer may be NULL. */
int skb_table_blocks(const skb_ctx *ctx, int32_t *on_demand, int32_t *blocks_last_call);

/* total kernels launched by this context so far (bench.py's gpu_launches) */
int64_t skb_launch_count(const skb_ctx *ctx);
/* device-side stopwatch: CUDA events recorded on the context's own stream */
int skb_timer_start(skb_ctx *ctx);
int skb_timer_stop(skb_ctx *ctx, float *ms);
/* CUDA stream the context launches on (cudaStream_t as void*), for external event timing */
void *skb_stream(const skb_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
