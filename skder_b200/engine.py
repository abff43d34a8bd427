"""Host-side mirror of the skani sub-commands skDER uses, on top of the C-ABI (include/skani_b200.h).

  skani sketch   -> Engine.add_fasta() + Engine.save()      (reference src/skDER/skder.py:103)
  skani triangle -> Engine.triangle()                       (skder.py:16-18)
  skani dist     -> Engine.rect(refs, queries)              (skder.py:58-59, cidder.py:362-363)
  skani search   -> Engine.load() + add query + rect()      (skder.py:119)

All compute happens in libskani_b200.so on the GPU; nothing here estimates anything.
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import SkbError

EDGE_DTYPE = np.dtype(
    {"names": ["a", "b", "ani", "af_a", "af_b"], "formats": ["<u4", "<u4", "<f8", "<f8", "<f8"],
     "offsets": [0, 4, 8, 16, 24], "itemsize": 32}
)
assert C.sizeof(_lib.Edge) == EDGE_DTYPE.itemsize
# skb_edge_detail: --detailed's per-edge record (Engine.last_edge_detail)
DETAIL_DTYPE = np.dtype(
    {"names": ["ani_lo", "ani_hi", "sd", "covered_a", "covered_b", "n_chains"],
     "formats": ["<f8", "<f8", "<f8", "<i8", "<i8", "<i4"], "offsets": [0, 8, 16, 24, 32, 40], "itemsize": 48}
)
assert C.sizeof(_lib.EdgeDetail) == DETAIL_DTYPE.itemsize


def default_params():
    p = _lib.Params()
    _lib.lib().skb_default_params(C.byref(p))
    return p


class PackedGenome:
    """2-bit packed genome in host memory (owned by the library)."""

    def __init__(self, ptr, path=None):
        self._p = ptr
        self.path = path

    def __del__(self):
        if getattr(self, "_p", None):
            _lib.lib().skb_packed_free(self._p)
            self._p = None

    n_bases = property(lambda s: s._p.contents.n_bases)
    n_words = property(lambda s: s._p.contents.n_words)
    n_contigs = property(lambda s: s._p.contents.n_contigs)
    n50 = property(lambda s: s._p.contents.n50)
    total_bases_all = property(lambda s: s._p.contents.total_bases_all)

    @property
    def first_name(self):
        return (self._p.contents.first_name or b"").decode("utf-8", "replace")

    @property
    def contig_names(self):
        """header lines (without '>') of the kept records, in file order; empty for pack_contigs' genomes"""
        names = self._p.contents.contig_names
        if not names:
            return []
        return [(names[k] or b"").decode("utf-8", "replace") for k in range(self.n_contigs)]

    def contig_lens(self):
        n = self.n_contigs
        return np.ctypeslib.as_array(self._p.contents.contig_lens, shape=(n,)).copy() if n else np.zeros(0, np.int64)

    def words(self):
        return np.ctypeslib.as_array(self._p.contents.words, shape=(self.n_words,))


def pack_fasta(path, min_contig_len=500):
    out = C.POINTER(_lib.Packed)()
    rc = _lib.lib().skb_pack_fasta(os.fsencode(path), min_contig_len, C.byref(out))
    if rc != 0 or not out:
        raise SkbError("cannot read FASTA %s (code %d)" % (path, rc))
    return PackedGenome(out, path)


def pack_fasta_many(paths, threads=None, min_contig_len=500):
    n = len(paths)
    if n == 0:
        return []
    arr = (C.c_char_p * n)(*[os.fsencode(p) for p in paths])
    out = (C.POINTER(_lib.Packed) * n)()
    threads = threads or os.cpu_count() or 1
    nfail = _lib.lib().skb_pack_fasta_many(arr, n, min_contig_len, threads, out)
    res = [PackedGenome(out[i], paths[i]) if out[i] else None for i in range(n)]
    if nfail:
        bad = [paths[i] for i in range(n) if res[i] is None]
        raise SkbError("cannot read %d FASTA file(s), first: %s" % (len(bad), bad[0]))
    return res


def pack_contigs(seqs, min_contig_len=500):
    seqs = [s if isinstance(s, bytes) else s.encode() for s in seqs]
    n = len(seqs)
    arr = (C.c_char_p * n)(*seqs)
    lens = (C.c_int64 * n)(*[len(s) for s in seqs])
    out = C.POINTER(_lib.Packed)()
    rc = _lib.lib().skb_pack_contigs(arr, lens, n, min_contig_len, C.byref(out))
    if rc != 0:
        raise SkbError("pack_contigs failed (code %d)" % rc)
    return PackedGenome(out)


def db_info(directory):
    """(genome count, marker compression m, 64-bit digest of the header and host tables) of directory/sketches.skb,
    read without a context or a device (skb_db_info)"""
    n, m, digest = C.c_int32(), C.c_int64(), C.c_uint64()
    rc = _lib.lib().skb_db_info(os.fsencode(directory), C.byref(n), C.byref(m), C.byref(digest))
    if rc != 0:
        raise SkbError("cannot read the sketch DB in %s (code %d)" % (directory, rc))
    return n.value, m.value, digest.value


class Engine:
    def __init__(self, device=0, params=None):
        self._L = _lib.lib()
        self._h = C.c_void_p()
        self.params = params or default_params()
        rc = self._L.skb_create(int(device), C.byref(self.params), C.byref(self._h))
        if rc != 0:
            raise SkbError("skb_create failed (%d): %s" % (rc, self._L.skb_last_error(None).decode()))
        self.device = int(device)
        self.detailed = False  # set_detailed
        self.last_query_contig_stats = None  # contig_stats of the last search's queries, with set_detailed(True)

    def close(self):
        if getattr(self, "_h", None):
            self._L.skb_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc, what):
        if rc != 0:
            raise SkbError("%s failed (%d): %s" % (what, rc, self._L.skb_last_error(self._h).decode()))

    ESTIMATORS = {"mean": 0, "median": 1, "robust": 2}  # SKB_ANI_MEAN / _MEDIAN / _ROBUST

    def set_estimator(self, name):
        """How a pair's accepted chains become one ANI in later triangle / rect / search / pairs calls: "mean" (skani's
        default), "median" (--median) or "robust" (--robust); DESIGN.md section 3.  Survives clear()."""
        if name not in self.ESTIMATORS:
            raise ValueError("unknown ANI estimator %r (mean, median, robust)" % (name,))
        self._ck(self._L.skb_set_ani_estimator(self._h, self.ESTIMATORS[name]), "skb_set_ani_estimator")

    def set_ci(self, on):
        """skani's --ci: later triangle / rect / search / pairs_edges calls also compute a bootstrap interval of every
        edge's ANI (last_edge_ci); DESIGN.md section 3.  Mean estimator only.  Survives clear()."""
        self._ck(self._L.skb_set_ani_ci(self._h, 1 if on else 0), "skb_set_ani_ci")

    def last_edge_ci(self):
        """(n, 2) float64 array: the 5th and 95th percentile ANI (percent) of every edge of the last triangle / rect /
        search / pairs_edges call, in edge order.  That call must have run with set_ci(True)."""
        ptr, n = C.POINTER(C.c_double)(), C.c_int64()
        self._ck(self._L.skb_last_edge_ci(self._h, C.byref(ptr), C.byref(n)), "skb_last_edge_ci")
        try:
            return np.ctypeslib.as_array(ptr, shape=(max(1, 2 * n.value),))[: 2 * n.value].reshape(n.value, 2).copy()
        finally:
            self._L.skb_free(ptr)

    def set_detailed(self, on):
        """skani's --detailed: later triangle / rect / search / pairs_edges calls also leave a detail record per edge
        (last_edge_detail), and search keeps the query's contig statistics (last_query_contig_stats); DESIGN.md section
        3.  Mean estimator only.  Survives clear()."""
        self._ck(self._L.skb_set_detailed(self._h, 1 if on else 0), "skb_set_detailed")
        self.detailed = bool(on)

    def last_edge_detail(self):
        """DETAIL_DTYPE array of every edge of the last triangle / rect / search / pairs_edges call, in edge order: the
        --ci interval and the chains' standard deviation (percent), the AF numerators of genomes a and b, the accepted
        chain count.  That call must have run with set_detailed(True)."""
        ptr, n = C.POINTER(_lib.EdgeDetail)(), C.c_int64()
        self._ck(self._L.skb_last_edge_detail(self._h, C.byref(ptr), C.byref(n)), "skb_last_edge_detail")
        try:
            if n.value == 0:
                return np.zeros(0, DETAIL_DTYPE)
            buf = C.cast(ptr, C.POINTER(C.c_char * (n.value * DETAIL_DTYPE.itemsize))).contents
            return np.frombuffer(buf, dtype=DETAIL_DTYPE, count=n.value).copy()
        finally:
            self._L.skb_free(ptr)

    def set_marker_compression(self, m):
        """skani's -m: genomes added from now on keep a canonical 21-mer as a marker iff its hash is below 2^64 // m
        (default 1000; DESIGN.md section 3).  Markers only decide which pairs pass the prescreen.  The context must be
        empty unless m is its current value; load() takes the database's m.  Survives clear()."""
        self._ck(self._L.skb_set_marker_compression(self._h, int(m)), "skb_set_marker_compression")

    def set_max_results(self, n):
        """skani's -n: later rect / search calls keep each query's first n edges in row order (ANI descending, ties to
        the lower reference id), with their last_edge_ci / last_edge_detail records; 0 (the default): all.  triangle and
        pairs_edges are unaffected.  DESIGN.md section 3.  Survives clear()."""
        self._ck(self._L.skb_set_max_results(self._h, int(n)), "skb_set_max_results")

    @property
    def marker_compression(self):
        m = C.c_int64()
        self._ck(self._L.skb_marker_compression(self._h, C.byref(m)), "skb_marker_compression")
        return m.value

    def contig_stats(self, first, n):
        """(n_contigs [n] int32, nx [n, 3] int64: N90, N50, N10) over the kept contigs of genomes first .. first+n-1"""
        cnt, nx = np.zeros(n, np.int32), np.zeros((n, 3), np.int64)
        self._ck(self._L.skb_genome_contig_stats(self._h, first, n, cnt.ctypes.data_as(C.POINTER(C.c_int32)),
                                                 nx.ctypes.data_as(C.POINTER(C.c_int64))), "skb_genome_contig_stats")
        return cnt, nx

    # ---- sketching -------------------------------------------------------------------------
    def add(self, packed, per_sequence=False):
        """Sketch packed genomes into the context.  per_sequence (skani's -i / --qi / --ri; DESIGN.md section 3): every
        kept record of every packed file becomes a genome of its own, ids in (file, record) order."""
        n = len(packed)
        if n == 0:
            return
        arr = (C.POINTER(_lib.Packed) * n)(*[p._p for p in packed])
        fn = "skb_add_sequences" if per_sequence else "skb_add_genomes"
        self._ck(getattr(self._L, fn)(self._h, n, arr), fn)

    def add_fasta(self, paths, threads=None):
        packed = pack_fasta_many(list(paths), threads, self.params.min_contig_len)
        self.add(packed)
        return packed

    def clear(self, keep_tables=False):
        if keep_tables:
            self._ck(self._L.skb_clear_keep_tables(self._h), "skb_clear_keep_tables")
        else:
            self._ck(self._L.skb_clear(self._h), "skb_clear")

    def index_seed_tables(self):
        self._ck(self._L.skb_index_seed_tables(self._h), "skb_index_seed_tables")

    def timer_start(self):
        self._ck(self._L.skb_timer_start(self._h), "skb_timer_start")

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self._L.skb_timer_stop(self._h, C.byref(ms)), "skb_timer_stop")
        return ms.value

    def index(self):
        self._ck(self._L.skb_index(self._h), "skb_index")

    def index_append(self):
        self._ck(self._L.skb_index_append(self._h), "skb_index_append")

    def pop_last_add(self):
        self._ck(self._L.skb_pop_last_add(self._h), "skb_pop_last_add")

    def search(self, query_packed, screen=80.0, min_af=15.0, per_sequence=False):
        """`skani search`: query genomes (one PackedGenome, or a list of them) against the resident, indexed database
        (ids 0..n-1), in one device pass.  The queries are sketched, indexed query-only, compared, and removed again.
        Edges: a = database genome, b = query (ids n, n+1, ... in list order).  per_sequence (skani's --qi): every kept
        record of the query files is a query, in (file, record) order.  With set_detailed(True) the queries'
        contig_stats are kept in last_query_contig_stats, in query order."""
        queries = list(query_packed) if isinstance(query_packed, (list, tuple)) else [query_packed]
        n_db = self.n_genomes
        self.add(queries, per_sequence)
        try:
            n_q = self.n_genomes - n_db
            if self.detailed:  # contig_stats of the queries: they leave the context below
                self.last_query_contig_stats = self.contig_stats(n_db, n_q)
            self.index_append()
            return self.rect(np.arange(n_db, dtype=np.int32), np.arange(n_db, n_db + n_q, dtype=np.int32),
                             screen=screen, min_af=min_af)
        finally:
            self.pop_last_add()

    @property
    def n_genomes(self):
        return self._L.skb_n_genomes(self._h)

    @property
    def launches(self):
        return self._L.skb_launch_count(self._h)

    def table_blocks(self):
        """(on_demand, blocks): whether the last index() chose on-demand seed tables -- the tables of all genomes exceed
        the table budget (SKB_TABLE_BUDGET_MB caps it) -- and how many blocks of tables the last triangle / rect / search /
        pairs_edges / pairs_detail call built (0 with resident tables).  DESIGN.md section 2."""
        on, blocks = C.c_int32(), C.c_int32()
        self._ck(self._L.skb_table_blocks(self._h, C.byref(on), C.byref(blocks)), "skb_table_blocks")
        return bool(on.value), int(blocks.value)

    @property
    def stream(self):
        return self._L.skb_stream(self._h)

    def sizes(self, g):
        ns, nm, tl = C.c_int64(), C.c_int64(), C.c_int64()
        nc = C.c_int32()
        self._ck(self._L.skb_sketch_sizes(self._h, g, C.byref(ns), C.byref(nm), C.byref(nc), C.byref(tl)), "skb_sketch_sizes")
        return {"n_seeds": ns.value, "n_markers": nm.value, "n_chunks": nc.value, "total_len": tl.value}

    def seeds(self, g):
        ns = C.c_int64()
        self._ck(self._L.skb_sketch_sizes(self._h, g, C.byref(ns), None, None, None), "skb_sketch_sizes")
        out = np.zeros(ns.value, np.uint64)
        self._ck(self._L.skb_get_seeds(self._h, g, out.ctypes.data), "skb_get_seeds")
        return out

    def markers(self, g):
        out = np.zeros(self.sizes(g)["n_markers"], np.uint64)
        self._ck(self._L.skb_get_markers(self._h, g, out.ctypes.data), "skb_get_markers")
        return out

    def save(self, directory):
        os.makedirs(directory, exist_ok=True)
        self._ck(self._L.skb_db_save(self._h, os.fsencode(directory)), "skb_db_save")

    def load(self, directory):
        self._ck(self._L.skb_db_load(self._h, os.fsencode(directory)), "skb_db_load")

    db_info = staticmethod(db_info)

    def load_genomes(self, directory, ids):
        """Append the database genomes `ids` (in that order) of `directory` as new genomes, bit-identical to adding
        their FASTAs (skb_db_load_genomes).  Before index(); one pop_last_add() undoes it."""
        ids = np.ascontiguousarray(ids, np.int32)
        self._ck(self._L.skb_db_load_genomes(self._h, os.fsencode(directory), ids.ctypes.data, len(ids)),
                 "skb_db_load_genomes")

    # ---- pairs -----------------------------------------------------------------------------
    def _take_edges(self, ptr, n):
        try:
            if n.value == 0:
                return np.zeros(0, EDGE_DTYPE)
            buf = C.cast(ptr, C.POINTER(C.c_char * (n.value * EDGE_DTYPE.itemsize))).contents
            return np.frombuffer(buf, dtype=EDGE_DTYPE, count=n.value).copy()
        finally:
            self._L.skb_free(ptr)

    def triangle(self, screen=80.0, min_af=15.0, part=0, n_parts=1, to_host=True):
        """to_host=False leaves the edges on the device (see device_edges) and returns (None, stats)."""
        ptr, n, st = C.POINTER(_lib.Edge)(), C.c_int64(), _lib.Stats()
        self._ck(
            self._L.skb_triangle(self._h, float(screen), float(min_af), part, n_parts,
                                 C.byref(ptr) if to_host else None, C.byref(n), C.byref(st)),
            "skb_triangle",
        )
        return (self._take_edges(ptr, n) if to_host else None), st

    def set_owned(self, first, count):
        """Seed tables are built (next index()) only for genomes first .. first+count-1; count = -1: all."""
        self._ck(self._L.skb_set_owned(self._h, int(first), int(count)), "skb_set_owned")

    def screen_triangle(self, screen=80.0, part=0, n_parts=1):
        """Prescreen of this partition's rows; returns (device pointer to the sorted (a << 32 | b) pairs, count, stats)."""
        ptr, n, st = C.c_void_p(), C.c_int64(), _lib.Stats()
        self._ck(self._L.skb_screen_triangle(self._h, float(screen), part, n_parts, C.byref(ptr), C.byref(n), C.byref(st)),
                 "skb_screen_triangle")
        return int(ptr.value or 0), int(n.value), st

    def pairs_edges(self, dev_pairs, n_pairs, owned_only=True, min_af=15.0, to_host=True):
        """ANI/AF of a device-resident pair list (only the pairs whose reference this context owns, if owned_only)."""
        ptr, n, st = C.POINTER(_lib.Edge)(), C.c_int64(), _lib.Stats()
        self._ck(
            self._L.skb_pairs_edges(self._h, C.c_void_p(dev_pairs), int(n_pairs), 1 if owned_only else 0, float(min_af),
                                    C.byref(ptr) if to_host else None, C.byref(n), C.byref(st)),
            "skb_pairs_edges",
        )
        return (self._take_edges(ptr, n) if to_host else None), st

    def greedy_summary(self, edges, n_genomes, min_ani, min_af):
        """(connectivity[n], member_off[n+1], members[]) of a binary edge list -- reference skDERsum's first pass.
        edges: EDGE_DTYPE array, or None for the list the last triangle/rect left on the device."""
        conn, off, mem = C.POINTER(C.c_int64)(), C.POINTER(C.c_int64)(), C.POINTER(C.c_uint32)()
        if edges is not None:
            edges = np.ascontiguousarray(edges, EDGE_DTYPE)
        self._ck(
            self._L.skb_greedy_summary(self._h, edges.ctypes.data if edges is not None else None,
                                       len(edges) if edges is not None else 0, int(n_genomes), float(min_ani), float(min_af),
                                       C.byref(conn), C.byref(off), C.byref(mem)),
            "skb_greedy_summary",
        )
        try:
            c = np.ctypeslib.as_array(conn, shape=(max(n_genomes, 1),))[:n_genomes].copy()
            o = np.ctypeslib.as_array(off, shape=(n_genomes + 1,)).copy()
            m = np.ctypeslib.as_array(mem, shape=(max(int(o[-1]), 1),))[: int(o[-1])].copy()
        finally:
            for p in (conn, off, mem):
                self._L.skb_free(p)
        return c, o, m

    MATRIX_KINDS = {"ani": 0, "distance": 1, "af": 2}  # SKB_MATRIX_ANI / _DISTANCE / _AF

    def write_matrix(self, path, labels, kind="ani", edges=None):
        """skani's --full-matrix files (DESIGN.md section 3), rendered on the device: "N\\n", then per genome its label
        and one tab-separated `%.2f` cell per genome.  kind "ani": the edge's ANI, 100.00 on the diagonal, 0.00 for no
        edge; "distance": 100.00 minus that cell's printed value; "af": the row genome's aligned fraction.  labels: one
        str (or bytes) per genome, in id order.  edges: EDGE_DTYPE array sorted by (a, b), or None for the list the last
        whole triangle() left on the device.  Writes `path` in place; the caller makes it atomic."""
        enc = [lb if isinstance(lb, bytes) else lb.encode("utf-8", "surrogateescape") for lb in labels]
        off = np.zeros(len(enc) + 1, np.int64)
        off[1:] = np.cumsum([len(x) for x in enc])
        if edges is not None:
            edges = np.ascontiguousarray(edges, EDGE_DTYPE)
        self._ck(
            self._L.skb_write_matrix(self._h, os.fsencode(path), self.MATRIX_KINDS[kind],
                                     edges.ctypes.data if edges is not None else None,
                                     len(edges) if edges is not None else 0, len(enc), b"".join(enc), off.ctypes.data),
            "skb_write_matrix",
        )

    def device_edges(self):
        """(device pointer, count) of the last triangle/rect result; valid until the next call on this engine."""
        ptr, n = C.c_void_p(), C.c_int64()
        self._ck(self._L.skb_device_edges(self._h, C.byref(ptr), C.byref(n)), "skb_device_edges")
        return int(ptr.value or 0), int(n.value)

    def rect(self, refs, queries, screen=80.0, min_af=15.0):
        refs = np.ascontiguousarray(refs, np.int32)
        queries = np.ascontiguousarray(queries, np.int32)
        ptr, n, st = C.POINTER(_lib.Edge)(), C.c_int64(), _lib.Stats()
        self._ck(
            self._L.skb_rect(self._h, refs.ctypes.data, len(refs), queries.ctypes.data, len(queries), float(screen),
                             float(min_af), C.byref(ptr), C.byref(n), C.byref(st)),
            "skb_rect",
        )
        return self._take_edges(ptr, n), st

    def pairs_detail(self, a, b):
        a = np.ascontiguousarray(a, np.uint32)
        b = np.ascontiguousarray(b, np.uint32)
        out = (_lib.PairDetail * len(a))()
        self._ck(self._L.skb_pairs_detail(self._h, a.ctypes.data, b.ctypes.data, len(a), out), "skb_pairs_detail")
        return out

    def shared_markers(self, a, b):
        a = np.ascontiguousarray(a, np.uint32)
        b = np.ascontiguousarray(b, np.uint32)
        out = np.zeros(len(a), np.int64)
        self._ck(self._L.skb_shared_markers(self._h, a.ctypes.data, b.ctypes.data, len(a), out.ctypes.data), "skb_shared_markers")
        return out

    def sketch_view(self):
        v = _lib.SketchView()
        self._ck(self._L.skb_sketch_view_get(self._h, C.byref(v)), "skb_sketch_view_get")
        return v
