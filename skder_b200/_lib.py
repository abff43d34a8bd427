"""ctypes view of include/skani_b200.h.  There is no Python or CPU implementation behind this
module: if libskani_b200.so is missing or no B200 is visible, calls fail loudly."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SKB_LIB") or os.path.join(HERE, "_lib", "libskani_b200.so")  # SKB_LIB: A/B builds


class SkbError(RuntimeError):
    pass


class Params(C.Structure):
    _fields_ = [
        ("min_contig_len", C.c_int32),
        ("chunk_len", C.c_int32),
        ("band_bp", C.c_int32),
        ("max_gap", C.c_int32),
        ("anchor_score", C.c_int32),
        ("min_anchors", C.c_int32),
        ("min_score", C.c_int32),
        ("max_mult", C.c_int32),
        ("max_chunk_chains", C.c_int32),
        ("ovl_num", C.c_int32),
        ("ovl_den", C.c_int32),
        ("span_ext", C.c_int32),
        ("debias_a", C.c_double),
        ("debias_g", C.c_double),
    ]


class Packed(C.Structure):
    _fields_ = [
        ("words", C.POINTER(C.c_uint64)),
        ("n_words", C.c_int64),
        ("n_bases", C.c_int64),
        ("n_contigs", C.c_int32),
        ("contig_lens", C.POINTER(C.c_int64)),
        ("first_name", C.c_char_p),
        ("n50", C.c_int64),
        ("total_bases_all", C.c_int64),
        ("contig_names", C.POINTER(C.c_char_p)),
    ]


class Edge(C.Structure):
    _fields_ = [("a", C.c_uint32), ("b", C.c_uint32), ("ani", C.c_double), ("af_a", C.c_double), ("af_b", C.c_double)]


class PairDetail(C.Structure):
    _fields_ = [
        ("a", C.c_uint32),
        ("b", C.c_uint32),
        ("ani", C.c_double),
        ("ani_raw", C.c_double),
        ("af_a", C.c_double),
        ("af_b", C.c_double),
        ("n_anchors", C.c_int64),
        ("n_seeds", C.c_int64),
        ("span_q", C.c_int64),
        ("span_r", C.c_int64),
        ("n_chains", C.c_int32),
        ("swapped", C.c_int32),
    ]


class EdgeDetail(C.Structure):  # skb_edge_detail
    _fields_ = [("ani_lo", C.c_double), ("ani_hi", C.c_double), ("sd", C.c_double), ("covered_a", C.c_int64),
                ("covered_b", C.c_int64), ("n_chains", C.c_int32), ("pad", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [
        ("n_pairs_total", C.c_int64),
        ("n_pairs_screened", C.c_int64),
        ("n_edges", C.c_int64),
        ("ms_screen", C.c_float),
        ("ms_ani", C.c_float),
        ("ms_total", C.c_float),
        ("launches", C.c_int64),
        ("sum_query_seeds", C.c_int64),
        ("sum_anchors", C.c_int64),
        ("ms_anchor", C.c_float),
        ("n_anchor_launches", C.c_int32),
    ]


class SketchView(C.Structure):
    _fields_ = [
        ("n_genomes", C.c_int32),
        ("n_seeds", C.c_int64),
        ("n_marker_keys", C.c_int64),
        ("n_contigs", C.c_int64),
        ("dev_seeds", C.c_void_p),
        ("dev_marker_keys", C.c_void_p),
        ("host_seed_off", C.POINTER(C.c_uint64)),
        ("host_total_len", C.POINTER(C.c_uint64)),
        ("host_ctg_off", C.POINTER(C.c_uint32)),
        ("host_ctg_len", C.POINTER(C.c_uint32)),
    ]


# every symbol include/skani_b200.h declares
SYMBOLS = [
    "skb_default_params", "skb_pack_fasta", "skb_pack_fasta_many", "skb_pack_contigs", "skb_packed_free",
    "skb_create", "skb_destroy", "skb_last_error", "skb_add_genomes", "skb_index", "skb_n_genomes",
    "skb_sketch_sizes", "skb_get_seeds", "skb_get_markers", "skb_db_save", "skb_db_load", "skb_triangle",
    "skb_rect", "skb_pairs_detail", "skb_shared_markers", "skb_sketch_view_get", "skb_import_sketches",
    "skb_free", "skb_launch_count", "skb_stream", "skb_clear", "skb_timer_start", "skb_timer_stop", "skb_index_append", "skb_pop_last_add",
    "skb_device_edges", "skb_set_owned", "skb_screen_triangle", "skb_pairs_edges", "skb_greedy_summary", "skb_index_seed_tables", "skb_clear_keep_tables",
    "skb_set_ani_estimator", "skb_set_ani_ci", "skb_last_edge_ci", "skb_set_detailed", "skb_last_edge_detail",
    "skb_genome_contig_stats", "skb_set_marker_compression", "skb_marker_compression", "skb_set_max_results",
    "skb_add_sequences",
]

_lib = None


def lib():
    """Load the shared library (never builds, never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SkbError(
            "libskani_b200.so not built (%s). Run `python -m skder_b200.build`; there is no CPU path." % LIB_PATH
        )
    L = C.CDLL(LIB_PATH)
    PP = C.POINTER(C.POINTER(Packed))
    L.skb_default_params.argtypes = [C.POINTER(Params)]
    L.skb_default_params.restype = None
    L.skb_pack_fasta.argtypes = [C.c_char_p, C.c_int32, PP]
    L.skb_pack_fasta_many.argtypes = [C.POINTER(C.c_char_p), C.c_int32, C.c_int32, C.c_int32, PP]
    L.skb_pack_contigs.argtypes = [C.POINTER(C.c_char_p), C.POINTER(C.c_int64), C.c_int32, C.c_int32, PP]
    L.skb_packed_free.argtypes = [C.POINTER(Packed)]
    L.skb_packed_free.restype = None
    L.skb_create.argtypes = [C.c_int32, C.POINTER(Params), C.POINTER(C.c_void_p)]
    L.skb_destroy.argtypes = [C.c_void_p]
    L.skb_destroy.restype = None
    L.skb_last_error.argtypes = [C.c_void_p]
    L.skb_last_error.restype = C.c_char_p
    L.skb_add_genomes.argtypes = [C.c_void_p, C.c_int32, PP]
    L.skb_add_sequences.argtypes = [C.c_void_p, C.c_int32, PP]
    L.skb_index.argtypes = [C.c_void_p]
    L.skb_n_genomes.argtypes = [C.c_void_p]
    L.skb_n_genomes.restype = C.c_int32
    L.skb_sketch_sizes.argtypes = [
        C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int64),
    ]
    L.skb_get_seeds.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.skb_get_markers.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    L.skb_db_save.argtypes = [C.c_void_p, C.c_char_p]
    L.skb_db_load.argtypes = [C.c_void_p, C.c_char_p]
    L.skb_triangle.argtypes = [
        C.c_void_p, C.c_double, C.c_double, C.c_int32, C.c_int32, C.POINTER(C.POINTER(Edge)), C.POINTER(C.c_int64),
        C.POINTER(Stats),
    ]
    L.skb_rect.argtypes = [
        C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_double, C.c_double,
        C.POINTER(C.POINTER(Edge)), C.POINTER(C.c_int64), C.POINTER(Stats),
    ]
    L.skb_pairs_detail.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(PairDetail)]
    L.skb_shared_markers.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    L.skb_sketch_view_get.argtypes = [C.c_void_p, C.POINTER(SketchView)]
    L.skb_import_sketches.argtypes = [
        C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
        C.c_void_p, C.c_int32,
    ]
    L.skb_set_owned.argtypes = [C.c_void_p, C.c_int32, C.c_int32]
    L.skb_screen_triangle.argtypes = [C.c_void_p, C.c_double, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                      C.POINTER(Stats)]
    L.skb_pairs_edges.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.POINTER(C.POINTER(Edge)),
                                  C.POINTER(C.c_int64), C.POINTER(Stats)]
    L.skb_greedy_summary.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_double,
                                     C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.POINTER(C.c_int64)), C.POINTER(C.POINTER(C.c_uint32))]
    L.skb_clear.argtypes = [C.c_void_p]
    L.skb_set_ani_estimator.argtypes = [C.c_void_p, C.c_int32]
    L.skb_set_ani_ci.argtypes = [C.c_void_p, C.c_int32]
    L.skb_set_detailed.argtypes = [C.c_void_p, C.c_int32]
    L.skb_last_edge_detail.argtypes = [C.c_void_p, C.POINTER(C.POINTER(EdgeDetail)), C.POINTER(C.c_int64)]
    L.skb_set_marker_compression.argtypes = [C.c_void_p, C.c_int64]
    L.skb_marker_compression.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
    L.skb_set_max_results.argtypes = [C.c_void_p, C.c_int64]
    L.skb_genome_contig_stats.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64)]
    L.skb_last_edge_ci.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_double)), C.POINTER(C.c_int64)]
    L.skb_index_seed_tables.argtypes = [C.c_void_p]
    L.skb_clear_keep_tables.argtypes = [C.c_void_p]
    L.skb_index_append.argtypes = [C.c_void_p]
    L.skb_pop_last_add.argtypes = [C.c_void_p]
    L.skb_timer_start.argtypes = [C.c_void_p]
    L.skb_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
    L.skb_free.argtypes = [C.c_void_p]
    L.skb_free.restype = None
    L.skb_launch_count.argtypes = [C.c_void_p]
    L.skb_launch_count.restype = C.c_int64
    L.skb_stream.argtypes = [C.c_void_p]
    L.skb_stream.restype = C.c_void_p
    _lib = L
    return L
