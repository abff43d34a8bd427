"""GPU parity: every stage of the CUDA path against the CPU oracle on identical inputs (through the C-ABI)."""
import itertools
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng7(built_lib, genomes7):
    from skder_b200 import engine

    e = engine.Engine(0)
    packed = e.add_fasta(genomes7, threads=4)
    e.index()
    yield e, packed
    e.close()


@pytest.fixture(scope="module")
def ora7(oracle, genomes7):
    return [oracle.Sketch.from_file(f) for f in genomes7]


def test_pack_matches_oracle_ingest(eng7, ora7):
    _, packed = eng7
    for p, s in zip(packed, ora7):
        assert p.n_bases == s.total_len
        assert p.n_contigs == s.n_contigs
        assert np.array_equal(p.contig_lens(), s.contig_lens())
        assert p.first_name == s.first_name


def test_seeds_bit_exact(eng7, ora7):
    e, _ = eng7
    for g, s in enumerate(ora7):
        mine, ref = e.seeds(g), s.seeds()
        assert len(mine) == len(ref), (g, len(mine), len(ref))
        assert np.array_equal(mine, ref), "genome %d: first diff at %d" % (g, int(np.argmax(mine != ref)))


def test_markers_bit_exact(eng7, ora7):
    e, _ = eng7
    for g, s in enumerate(ora7):
        assert np.array_equal(e.markers(g), s.markers())
        assert e.sizes(g)["n_chunks"] == s.n_chunks


def test_shared_marker_counts_bit_exact(eng7, ora7, oracle):
    e, _ = eng7
    pairs = list(itertools.combinations(range(7), 2))
    a = [p[0] for p in pairs]
    b = [p[1] for p in pairs]
    got = e.shared_markers(a, b)
    want = [oracle.screen(ora7[i], ora7[j], 0.8)[0] for i, j in pairs]
    assert list(got) == want


def test_pairs_integer_exact_and_float_close(eng7, ora7, oracle):
    e, _ = eng7
    pairs = list(itertools.combinations(range(7), 2)) + [(3, 1), (6, 0)]
    det = e.pairs_detail([p[0] for p in pairs], [p[1] for p in pairs])
    for (i, j), d in zip(pairs, det):
        r = oracle.pair(ora7[i], ora7[j])
        assert (d.swapped, d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r) == (
            r.swapped, r.n_chains, r.n_anchors_total, r.n_seeds_total, r.span_q, r.span_r), (i, j)
        # tolerance: same IEEE expressions; device pow() vs glibc pow() may differ in the last ulps
        assert abs(d.ani_raw - r.ani_raw) < 1e-12 and abs(d.ani - r.ani) < 1e-12
        assert abs(d.af_a - r.af_a) < 1e-15 and abs(d.af_b - r.af_b) < 1e-15


def test_triangle_screen_and_edges(eng7, ora7, oracle):
    e, _ = eng7
    edges, st = e.triangle(screen=89.0, min_af=50.0)
    want = {}
    for i, j in itertools.combinations(range(7), 2):
        if not oracle.screen(ora7[i], ora7[j], 0.89)[1]:
            continue
        r = oracle.pair(ora7[i], ora7[j])
        if r.ani >= 0 and max(r.af_a, r.af_b) * 100 >= 50.0:
            want[(i, j)] = ("%.2f" % (r.ani * 100), "%.2f" % (r.af_a * 100), "%.2f" % (r.af_b * 100))
    got = {(int(x["a"]), int(x["b"])): ("%.2f" % x["ani"], "%.2f" % x["af_a"], "%.2f" % x["af_b"]) for x in edges}
    assert got == want
    assert st.n_pairs_total == 21 and st.n_edges == len(want)
    # a screen nobody passes -> no pairs, no edges
    edges2, st2 = e.triangle(screen=99.999, min_af=0.0)
    none_pass = not any(oracle.screen(ora7[i], ora7[j], 0.99999)[1] for i, j in itertools.combinations(range(7), 2))
    if none_pass:
        assert len(edges2) == 0 and st2.n_pairs_screened == 0


def test_triangle_partitions_cover_triangle(eng7):
    e, _ = eng7
    full, _ = e.triangle(screen=80.0, min_af=0.0)
    from skder_b200 import multi

    for n_parts in (2, 3, 5):
        parts = []
        for p in range(n_parts):
            edges, st = e.triangle(screen=0.0, min_af=0.0, part=p, n_parts=n_parts)
            rows, npairs = multi.partition_rows(7, p, n_parts)  # the host-side statement of the same dealing rule
            assert st.n_pairs_total == npairs and set(edges["a"].tolist()) <= set(rows.tolist())
            parts.append(e.triangle(screen=80.0, min_af=0.0, part=p, n_parts=n_parts)[0])
        cat = np.sort(np.concatenate(parts), order=["a", "b"])
        assert np.array_equal(cat, np.sort(full, order=["a", "b"]))


def test_rect_equals_triangle_values(eng7):
    e, _ = eng7
    tri, _ = e.triangle(screen=80.0, min_af=0.0)
    tv = {(int(x["a"]), int(x["b"])): (x["ani"], x["af_a"], x["af_b"]) for x in tri}
    refs, queries = [0, 2, 5, 6], [1, 3, 4]
    rect, st = e.rect(refs, queries, screen=80.0, min_af=0.0)
    assert st.n_pairs_total == 12
    for x in rect:
        a, b = int(x["a"]), int(x["b"])
        assert a in refs and b in queries
        if a < b:
            assert tv[(a, b)] == (x["ani"], x["af_a"], x["af_b"])
        else:  # same estimator, roles swapped back
            assert tv[(b, a)] == (x["ani"], x["af_b"], x["af_a"])
    assert len(rect) == 12


# the automatic seed-table density, and two records per 4-slot bucket (SKB_TAB_X2=1), which fills overflow chains
@pytest.mark.parametrize("tab_x2", [None, "1"], ids=["auto", "SKB_TAB_X2=1"])
def test_appended_index_equals_full_index(genomes7, built_lib, monkeypatch, tab_x2):
    """Genomes indexed by skb_index_append get the chunk tables, marker lists and per-pair results a full skb_index gives
    them, and popping them leaves the database as it was."""
    from skder_b200 import engine

    if tab_x2:
        monkeypatch.setenv("SKB_TAB_X2", tab_x2)
    else:
        monkeypatch.delenv("SKB_TAB_X2", raising=False)
    packed = engine.pack_fasta_many(genomes7, threads=4)
    with engine.Engine(0) as app, engine.Engine(0) as full:
        app.add(packed[:5])
        app.index()
        app.add([packed[5]])
        app.add([packed[6]])
        app.index_append()
        full.add(packed)
        full.index()
        for g in (5, 6):
            assert app.sizes(g) == full.sizes(g)
            assert np.array_equal(app.markers(g), full.markers(g))
        assert app.rect(range(5), [5, 6])[0].tobytes() == full.rect(range(5), [5, 6])[0].tobytes()
        pairs = [p for g in (5, 6) for x in range(5) for p in ((x, g), (g, x))]
        a, b = [p[0] for p in pairs], [p[1] for p in pairs]
        for p, x, y in zip(pairs, app.pairs_detail(a, b), full.pairs_detail(a, b)):
            assert bytes(x) == bytes(y), p  # integers and doubles bit for bit
        app.pop_last_add()
        app.pop_last_add()
        with engine.Engine(0) as db:
            db.add(packed[:5])
            db.index()
            assert app.triangle(min_af=0.0)[0].tobytes() == db.triangle(min_af=0.0)[0].tobytes()
    # a context that owns genomes 0-4 builds no seed table for an appended genome, and refuses it as a reference
    with engine.Engine(0) as part:
        part.add(packed[:5])
        part.set_owned(0, 5)
        part.index()
        part.add([packed[5]])
        part.index_append()
        ns = [part.sizes(g)["n_seeds"] for g in range(6)]
        for x in range(5):
            a, b = (x, 5) if ns[5] >= ns[x] else (5, x)  # the reference is the genome with more seeds (ties: b)
            with pytest.raises(engine.SkbError):
                part.pairs_detail([a], [b])


def test_db_roundtrip(eng7, tmp_path):
    from skder_b200 import engine

    e, _ = eng7
    e.save(str(tmp_path))
    with engine.Engine(0) as e2:
        e2.load(str(tmp_path))
        e2.index()
        assert e2.n_genomes == 7
        for g in range(7):
            assert np.array_equal(e.seeds(g), e2.seeds(g))
            assert np.array_equal(e.markers(g), e2.markers(g))
        t1, _ = e.triangle(80.0, 0.0)
        t2, _ = e2.triangle(80.0, 0.0)
        assert np.array_equal(t1, t2)


def test_synthetic_clades(oracle, built_lib):
    from skder_b200 import engine, synth

    gens = [c for _, _, c in synth.config_genomes("tiny")]
    sk = [oracle.Sketch.from_contigs(c) for c in gens]
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(c) for c in gens])
        e.index()
        for g, s in enumerate(sk):
            assert np.array_equal(e.seeds(g), s.seeds())
            assert np.array_equal(e.markers(g), s.markers())
        edges, st = e.triangle(screen=80.0, min_af=15.0)
        n = len(gens)
        want = {}
        for i, j in itertools.combinations(range(n), 2):
            if not oracle.screen(sk[i], sk[j], 0.80)[1]:
                continue
            r = oracle.pair(sk[i], sk[j])
            if r.ani >= 0 and max(r.af_a, r.af_b) * 100 >= 15.0:
                want[(i, j)] = ("%.2f" % (r.ani * 100), "%.2f" % (r.af_a * 100), "%.2f" % (r.af_b * 100))
        got = {(int(x["a"]), int(x["b"])): ("%.2f" % x["ani"], "%.2f" % x["af_a"], "%.2f" % x["af_b"]) for x in edges}
        assert got == want
        # 3 clades x 4: only within-clade pairs survive
        assert len(want) == 3 * 6


def _run_shim(argv):
    import subprocess
    import sys

    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "skder_b200", "bin", "skani")
    return subprocess.call([sys.executable, shim] + argv, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def test_skani_shim_triangle_dist_search_bytes_equal_oracle(genomes7, oracle, built_lib, tmp_path):
    """The `skani` stand-in, invoked exactly as skDER spells it (reference src/skDER/skder.py:16-18, 58-59, 103, 119),
    writes byte-for-byte the TSV the CPU oracle writes."""
    from oracle import skani_cpu

    lst = tmp_path / "All_Genomes_Listing.txt"
    lst.write_text("".join(p + "\n" for p in reversed(genomes7)))  # list order must not matter
    out = tmp_path / "Skani_Triangle_Edge_Output.txt"
    assert _run_shim(["triangle", "-l", str(lst), "--min-af", "50.0", "-E", "-s", "89.0", "-t", "4", "-o", str(out)]) == 0
    assert out.read_text() == skani_cpu.triangle_tsv(genomes7, 89.0, 50.0, threads=4)
    # provenance beside the output: skDER discards stdout/stderr, and the numbers are not the skani binary's
    assert "NOT the skani binary" in (tmp_path / (out.name + ".skani_b200.log")).read_text()
    # dist: reps vs non-reps, no -t, default screen / min-af
    rl, ql = tmp_path / "Reps_Listing.txt", tmp_path / "NonReps_Listing.txt"
    rl.write_text("".join(p + "\n" for p in genomes7[:4]))
    ql.write_text("".join(p + "\n" for p in genomes7[4:]))
    dout = tmp_path / "Skani_Dist_Output.txt"
    assert _run_shim(["dist", "--rl", str(rl), "--ql", str(ql), "-s", "89.0", "-o", str(dout)]) == 0
    assert dout.read_text() == skani_cpu.rect_tsv(genomes7[:4], genomes7[4:], 89.0, 15.0, threads=4)
    # sketch + search (low_mem_greedy): DB directory, then one query against it
    db = tmp_path / "skani_sketch_all.db"
    assert _run_shim(["sketch", "-l", str(lst), "-o", str(db), "-t", "4"]) == 0 and db.is_dir()
    sout = tmp_path / "current_search_results.tsv"
    q = genomes7[2]
    from skder_b200 import daemon

    try:
        assert _run_shim(["search", q, "-d", str(db), "-o", str(sout), "-t", "4"]) == 0
    finally:
        daemon.stop_for(str(db))  # the search started the database's server: it must not outlive the test
    rows = [ln.split("\t") for ln in sout.read_text().splitlines()[1:]]
    assert len(rows) == 7 and all(r[1] == q for r in rows)  # 6 partners + the genome's own copy in the DB
    self_row = [r for r in rows if r[0] == q][0]
    assert self_row[2] == "100.00" and float(self_row[3]) > 99.5
    sk = {p: oracle.Sketch.from_file(p) for p in genomes7}
    for r in rows:
        res = oracle.pair(sk[r[0]], sk[q]) if r[0] != q else None
        if res is not None:
            assert (r[2], r[3], r[4]) == ("%.2f" % (res.ani * 100), "%.2f" % (res.af_a * 100), "%.2f" % (res.af_b * 100))
    assert [float(r[2]) for r in rows] == sorted((float(r[2]) for r in rows), reverse=True)  # ANI descending
    # unsupported option: non-zero exit and the previous output is not replaced by a partial file
    bad = tmp_path / "bad.tsv"
    assert _run_shim(["triangle", "-l", str(lst), "-E", "--medium", "-o", str(bad)]) != 0 and not bad.exists()


def test_full_size_properties(built_lib):
    """BASELINE config-sized genomes (5 Mbp): size-independent properties through the C-ABI."""
    from skder_b200 import engine, synth

    gens = [engine.pack_contigs(c) for c in synth.one_clade(0, 6, 5_000_000, 99)] + \
           [engine.pack_contigs(c) for c in synth.one_clade(1, 2, 5_000_000, 99)]
    with engine.Engine(0) as e:
        e.add(gens)
        e.add([gens[0]])  # an exact copy of genome 0 becomes genome 8
        e.index()
        edges, st = e.triangle(screen=80.0, min_af=15.0)
        got = {(int(x["a"]), int(x["b"])): x for x in edges}
        # within-clade pairs only; cross-clade pairs die in the prescreen
        clade = lambda g: 0 if g < 6 or g == 8 else 1
        assert all(clade(a) == clade(b) for a, b in got) and len(got) == 21 + 1
        assert st.n_pairs_total == 36 and st.n_pairs_screened == 22
        # idempotence: a genome against its copy is 100 / ~100 / ~100
        x = got[(0, 8)]
        assert x["ani"] == 100.0 and x["af_a"] > 99.5 and x["af_b"] > 99.5  # chain ends are clipped to chunk bounds
        # the copy behaves exactly like the original against everyone else
        for b in range(1, 6):
            assert (got[(0, b)]["ani"], got[(0, b)]["af_a"]) == (got[(b, 8)]["ani"], got[(b, 8)]["af_b"])
        # ANI decreases with the mutation rates that generated the clade (d_i + d_j), within sampling noise
        d = e.pairs_detail([0, 0], [1, 2])
        assert all(0.90 < x.ani_raw < 1.0 for x in d)
        # sketch density at full size
        for g in range(8):
            s = e.sizes(g)
            assert abs(s["n_seeds"] / (s["total_len"] / 125.0) - 1) < 0.03


def test_edge_cases_through_the_abi(oracle, built_lib):
    """empty / tiny / all-N genomes, single genome, re-index after adding, clear and reuse, bad arguments"""
    from skder_b200 import engine

    rng = np.random.default_rng(5)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    big = bytes(acgt[rng.integers(0, 4, 120_000)])
    mut = bytearray(big)
    for p in rng.integers(0, len(mut), 1200):
        mut[p] = b"ACGT"[(b"ACGT".index(mut[p]) + 1) % 4]
    contig_sets = [
        [],                                   # no contigs at all
        [b"ACGTTGCA" * 50],                   # 400 bp: below min_contig_len, dropped
        [b"N" * 3000],                        # packs as poly-A
        [big],
        [bytes(mut[:50_000]), bytes(mut[50_000:])],
        [b"acgt" * 200 + big[:5000].lower()],  # lowercase
    ]
    sk = [oracle.Sketch.from_contigs(c) for c in contig_sets]
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(contig_sets[3])])
        e.index()
        edges, st = e.triangle(80.0, 0.0)  # a single genome: no pairs
        assert len(edges) == 0 and st.n_pairs_total == 0
        with pytest.raises(engine.SkbError):
            e.pairs_detail([0], [0])
        with pytest.raises(engine.SkbError):
            e.rect([0], [5])
        e.clear()
        assert e.n_genomes == 0
        with pytest.raises(engine.SkbError):
            e.index()  # nothing to index
        e.add([engine.pack_contigs(c) for c in contig_sets[:4]])
        with pytest.raises(engine.SkbError):
            e.triangle(80.0, 0.0)  # not indexed yet
        e.index()
        e.add([engine.pack_contigs(c) for c in contig_sets[4:]])  # more genomes after an index
        with pytest.raises(engine.SkbError):
            e.triangle(80.0, 0.0)  # stale index is refused
        e.index()
        assert e.n_genomes == 6
        for g, s in enumerate(sk):
            assert np.array_equal(e.seeds(g), s.seeds()), g
            assert np.array_equal(e.markers(g), s.markers()), g
            assert e.sizes(g)["n_chunks"] == s.n_chunks and e.sizes(g)["total_len"] == s.total_len
        pairs = list(itertools.combinations(range(6), 2))
        det = e.pairs_detail([p[0] for p in pairs], [p[1] for p in pairs])
        for (i, j), d in zip(pairs, det):
            r = oracle.pair(sk[i], sk[j])
            assert (d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r) == (
                r.n_chains, r.n_anchors_total, r.n_seeds_total, r.span_q, r.span_r), (i, j)
            assert (d.ani < 0) == (r.ani < 0)
            if r.ani >= 0:
                assert abs(d.ani - r.ani) < 1e-12
        got = e.shared_markers([p[0] for p in pairs], [p[1] for p in pairs])
        assert list(got) == [oracle.screen(sk[i], sk[j], 0.8)[0] for i, j in pairs]
        # screening off (-s 0): every pair is evaluated; only pairs with an estimate become edges
        edges, st = e.triangle(0.0, 0.0)
        assert st.n_pairs_screened == 15
        want = {(i, j) for i, j in pairs if oracle.pair(sk[i], sk[j]).ani >= 0}
        assert {(int(x["a"]), int(x["b"])) for x in edges} == want and (3, 4) in want
        # empty id lists
        edges, st = e.rect([], [1, 2])
        assert len(edges) == 0


def test_engine_search_and_daemon(genomes7, oracle, built_lib, tmp_path, monkeypatch):
    """`skani search` three ways -- Engine.search on a resident DB, the shim in-process (SKB_NO_DAEMON=1) and the
    shim through the resident daemon, twice -- all give the oracle's rows; the DB is untouched afterwards."""
    import subprocess
    import sys

    from oracle import skani_cpu
    from skder_b200 import daemon, engine

    lst = tmp_path / "list.txt"
    lst.write_text("".join(p + "\n" for p in genomes7))
    db = tmp_path / "db"
    assert _run_shim(["sketch", "-l", str(lst), "-o", str(db), "-t", "4"]) == 0
    sk = {p: oracle.Sketch.from_file(p) for p in genomes7}

    def want_rows(q):
        rows = []
        for r in genomes7:
            res = oracle.pair(sk[r], sk[q])
            if oracle.screen(sk[r], sk[q], 0.8)[1] and res.ani >= 0 and max(res.af_a, res.af_b) >= 0.15:
                rows.append((r, "%.2f" % (res.ani * 100), "%.2f" % (res.af_a * 100), "%.2f" % (res.af_b * 100)))
        return sorted(rows)

    with engine.Engine(0) as e:
        e.load(str(db))
        e.index()
        before, _ = e.triangle(80.0, 0.0)
        for q in (genomes7[1], genomes7[5]):
            edges, st = e.search(engine.pack_fasta(q))
            got = sorted((genomes7[int(x["a"])], "%.2f" % x["ani"], "%.2f" % x["af_a"], "%.2f" % x["af_b"]) for x in edges)
            assert got == want_rows(q) and all(int(x["b"]) == 7 for x in edges)
            assert e.n_genomes == 7
        after, _ = e.triangle(80.0, 0.0)
        assert np.array_equal(before, after)  # the query came and went; the database is unchanged

    def rows_of(path):
        return sorted((t[0], t[2], t[3], t[4]) for t in (ln.split("\t") for ln in open(path).read().splitlines()[1:]))

    out = tmp_path / "s.tsv"
    monkeypatch.setenv("SKB_NO_DAEMON", "1")
    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "skder_b200", "bin", "skani")
    assert subprocess.call([sys.executable, shim, "search", genomes7[3], "-d", str(db), "-o", str(out), "-t", "2"]) == 0
    assert rows_of(out) == want_rows(genomes7[3])
    monkeypatch.delenv("SKB_NO_DAEMON")
    monkeypatch.setenv("SKB_DAEMON_IDLE", "120")
    try:
        for q in (genomes7[0], genomes7[6], genomes7[0]):
            out.unlink()
            assert subprocess.call([sys.executable, shim, "search", q, "-d", str(db), "-o", str(out), "-t", "2"]) == 0
            assert rows_of(out) == want_rows(q)
        assert daemon.request(str(db), 0, {"op": "ping"}, timeout=5.0)["n"] == 7  # one server answered all three
        # the socket is private and authenticated: mode 0600 in a 0700 directory, key 0600 inside the database
        import stat

        sock = daemon.socket_path(str(db), 0)
        assert stat.S_IMODE(os.stat(sock).st_mode) == 0o600 and stat.S_IMODE(os.stat(os.path.dirname(sock)).st_mode) == 0o700
        assert stat.S_IMODE(os.stat(daemon._key_path(str(db), 0)).st_mode) == 0o600
        # a re-run sketches a DIFFERENT genome set into the same directory (skDER reuses its output directory): the next
        # search must be answered from the new database, never from the resident copy of the old one
        lst.write_text("".join(p + "\n" for p in genomes7[:5]))
        assert _run_shim(["sketch", "-l", str(lst), "-o", str(db), "-t", "4"]) == 0
        out.unlink()
        assert subprocess.call([sys.executable, shim, "search", genomes7[0], "-d", str(db), "-o", str(out), "-t", "2"]) == 0
        assert {r[0] for r in rows_of(out)} <= set(genomes7[:5]) and len(rows_of(out)) == 5
        assert daemon.request(str(db), 0, {"op": "ping"}, timeout=5.0)["n"] == 5
        # ... and when the files are swapped behind a running server's back (no `skani sketch` of ours involved)
        import shutil

        other = tmp_path / "db2"
        lst.write_text("".join(p + "\n" for p in genomes7[2:]))
        assert _run_shim(["sketch", "-l", str(lst), "-o", str(other), "-t", "4"]) == 0
        for f in ("sketches.skb", "manifest.json"):
            shutil.copyfile(other / f, db / (f + ".new"))
            os.replace(db / (f + ".new"), db / f)
        out.unlink()
        assert subprocess.call([sys.executable, shim, "search", genomes7[6], "-d", str(db), "-o", str(out), "-t", "2"]) == 0
        assert {r[0] for r in rows_of(out)} <= set(genomes7[2:]) and len(rows_of(out)) == 5
    finally:
        daemon.stop_for(str(db))


def test_many_chains_in_one_chunk(oracle, built_lib):
    """A query chunk stitched from 14 distant reference segments: more qualifying DP trees than chain_kernel tracks
    in registers (fallback to ends_kernel) and more chains than slots per chunk (top-8 selection); plus a
    tandem-duplicated reference (several hits per seed: staging, sort by reference position, multiplicity cap)."""
    from skder_b200 import engine

    rng = np.random.default_rng(11)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    ref = acgt[rng.integers(0, 4, 400_000)]
    order = rng.permutation(14)
    query = np.concatenate([ref[20_000 * (k + 1): 20_000 * (k + 1) + 1300] for k in order] + [acgt[rng.integers(0, 4, 30_000)]])
    unit = acgt[rng.integers(0, 4, 6_000)]
    tandem = np.concatenate([unit] * 5 + [acgt[rng.integers(0, 4, 50_000)]])  # every k-mer of `unit` 5x
    tandem_q = np.concatenate([acgt[rng.integers(0, 4, 3_000)], unit, acgt[rng.integers(0, 4, 3_000)]])
    sets = [[ref.tobytes()], [query.tobytes()], [tandem.tobytes()], [tandem_q.tobytes()]]
    sk = [oracle.Sketch.from_contigs(c) for c in sets]
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(c) for c in sets])
        e.index()
        det = e.pairs_detail([0, 2], [1, 3])
        for (i, j), d in zip([(0, 1), (2, 3)], det):
            r = oracle.pair(sk[i], sk[j])
            assert (d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r, d.swapped) == (
                r.n_chains, r.n_anchors_total, r.n_seeds_total, r.span_q, r.span_r, r.swapped), (i, j)
            assert abs(d.ani - r.ani) < 1e-12 and abs(d.af_a - r.af_a) < 1e-15
        assert det[0].n_chains == 8  # 14 chains in the first query chunk, 8 slots
        assert det[1].n_chains >= 1 and det[1].n_anchors > 0


def test_device_edges_match_host_copy(eng7):
    """skb_device_edges: the device-resident result (multi-GPU gather path) equals the host copy, with and without
    the host copy being made."""
    import torch

    from skder_b200 import multi
    from skder_b200.engine import EDGE_DTYPE

    e, _ = eng7
    host, st = e.triangle(screen=80.0, min_af=0.0)
    for to_host in (True, False):
        got, st2 = e.triangle(screen=80.0, min_af=0.0, to_host=to_host)
        assert (got is None) == (not to_host) and st2.n_edges == len(host)
        ptr, n = e.device_edges()
        assert n == len(host)
        dev = multi._dev_tensor(torch, ptr, n * (EDGE_DTYPE.itemsize // 8), torch.device("cuda", e.device))
        assert np.array_equal(dev.cpu().numpy().view(EDGE_DTYPE), host)


def test_general_and_narrow_pair_kernels_agree(eng7, monkeypatch):
    """anchor_kernel / chain_kernel come in two variants: 32-bit record matching and diagonal arithmetic when every
    padded position is below 2^30 (what any bacterial set runs), and the general one.  SKB_WIDE_DIAG=1 forces the
    general variants: every integer and float of every pair must be identical."""
    e, _ = eng7
    pairs = list(itertools.combinations(range(7), 2)) + [(3, 1), (6, 0)]
    a, b = [p[0] for p in pairs], [p[1] for p in pairs]
    monkeypatch.delenv("SKB_WIDE_DIAG", raising=False)
    narrow = e.pairs_detail(a, b)
    monkeypatch.setenv("SKB_WIDE_DIAG", "1")
    wide = e.pairs_detail(a, b)
    key = lambda d: (d.swapped, d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r, d.ani_raw, d.ani, d.af_a, d.af_b)
    assert [key(d) for d in narrow] == [key(d) for d in wide]
    assert any(d.n_chains > 0 for d in narrow)


def test_full_size_genomes_against_oracle(oracle, built_lib):
    """BASELINE config-sized genomes (10 x 5 Mbp: two clades of 4 and two singletons) against the oracle, through the
    C-ABI: sketches bit-exact, prescreen decisions equal, pair integers exact, the 2-decimal edge list identical."""
    from skder_b200 import engine, synth

    sets = synth.one_clade(0, 4, 5_000_000, 1234) + synth.one_clade(1, 4, 5_000_000, 1234) + \
        synth.one_clade(2, 1, 5_000_000, 1234) + synth.one_clade(3, 1, 5_000_000, 1234)
    sk = [oracle.Sketch.from_contigs(c) for c in sets]
    n = len(sets)
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(c) for c in sets])
        e.index()
        for g, s in enumerate(sk):
            assert np.array_equal(e.seeds(g), s.seeds()), g
            assert np.array_equal(e.markers(g), s.markers()), g
        pairs = list(itertools.combinations(range(n), 2))
        shared = e.shared_markers([p[0] for p in pairs], [p[1] for p in pairs])
        scr = [oracle.screen(sk[i], sk[j], 0.895) for i, j in pairs]
        assert list(shared) == [x[0] for x in scr]
        edges, st = e.triangle(screen=89.5, min_af=50.0)
        assert st.n_pairs_screened == sum(x[1] for x in scr) == 12
        surv = [p for p, x in zip(pairs, scr) if x[1]]
        det = e.pairs_detail([p[0] for p in surv], [p[1] for p in surv])
        want = {}
        for (i, j), d in zip(surv, det):
            r = oracle.pair(sk[i], sk[j])
            assert (d.swapped, d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r) == (
                r.swapped, r.n_chains, r.n_anchors_total, r.n_seeds_total, r.span_q, r.span_r), (i, j)
            assert abs(d.ani - r.ani) < 1e-12 and abs(d.af_a - r.af_a) < 1e-15 and abs(d.af_b - r.af_b) < 1e-15
            if r.ani >= 0 and max(r.af_a, r.af_b) * 100 >= 50.0:
                want[(i, j)] = ("%.2f" % (r.ani * 100), "%.2f" % (r.af_a * 100), "%.2f" % (r.af_b * 100))
        got = {(int(x["a"]), int(x["b"])): ("%.2f" % x["ani"], "%.2f" % x["af_a"], "%.2f" % x["af_b"]) for x in edges}
        assert got == want and len(want) == 12


def test_fragmented_genome_beyond_the_shared_memory_limits(oracle, built_lib):
    """A MAG-like query of 6,000 contigs (one chunk and one chain each: more chunks and more chain candidates than
    the shared-memory finalize kernel takes) against its unfragmented source, next to ordinary pairs in the same call:
    the pair runs on the global-memory instance, the call succeeds, everything equals the oracle."""
    from skder_b200 import engine

    rng = np.random.default_rng(21)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    whole = acgt[rng.integers(0, 4, 6000 * 800)]
    frag = [whole[k * 800:(k + 1) * 800].tobytes() for k in range(6000)]
    other = bytearray(whole[:400_000].tobytes())
    for p in rng.integers(0, len(other), 4000):
        other[p] = b"ACGT"[(b"ACGT".index(other[p]) + 1) % 4]
    sets = [[whole.tobytes()], frag, [bytes(other)]]
    sk = [oracle.Sketch.from_contigs(c) for c in sets]
    assert sk[1].n_chunks == 6000
    with engine.Engine(0) as e:
        e.add([engine.pack_contigs(c) for c in sets])
        e.index()
        pairs = [(0, 1), (0, 2), (1, 2)]
        det = e.pairs_detail([p[0] for p in pairs], [p[1] for p in pairs])
        for (i, j), d in zip(pairs, det):
            r = oracle.pair(sk[i], sk[j])
            assert (d.swapped, d.n_chains, d.n_anchors, d.n_seeds, d.span_q, d.span_r) == (
                r.swapped, r.n_chains, r.n_anchors_total, r.n_seeds_total, r.span_q, r.span_r), (i, j)
            assert abs(d.ani - r.ani) < 1e-12 and abs(d.af_a - r.af_a) < 1e-15 and abs(d.af_b - r.af_b) < 1e-15
        assert det[0].n_chains > 4096 and det[0].swapped == 1  # the fragmented copy is the query
        edges, st = e.triangle(screen=80.0, min_af=15.0)
        assert len(edges) == 3


def test_binary_edge_handoff_equals_reference_skdersum(eng7, genomes7, built_lib, tmp_path):
    """SURVEY section 8 f3: Genome_Information_for_Greedy_Clustering.txt from binary edges (skb_greedy_summary + select.py) is
    byte-identical to what the reference's skDERsum prints from the TSV (tests/replay.py, held to the reference's own
    output by the CPU tests) -- on both golden edge lists (ids assigned from their paths) and on this engine's own
    unrounded edges against its own TSV."""
    import replay
    from conftest import GOLDEN
    from skder_b200 import cli, select
    from skder_b200.engine import EDGE_DTYPE

    e, packed = eng7
    for gdir, cuts in (("skder_results", [(99.0, 50.0), (97.0, 50.0)]), ("skder_gtdb_results", [(99.0, 50.0), (98.0, 90.0), (90.0, 10.0)])):
        tsv = os.path.join(GOLDEN, gdir, "Skani_Triangle_Edge_Output.txt")
        n50f = os.path.join(GOLDEN, gdir, "Concatenated_N50.txt")
        rows = [ln.rstrip("\n").split("\t") for ln in open(tsv).read().splitlines()[1:]]
        paths = sorted({r[0] for r in rows} | {r[1] for r in rows} | {ln.split("\t")[0] for ln in open(n50f) if ln.strip()})
        idx = {p: i for i, p in enumerate(paths)}
        edges = np.array([(idx[r[0]], idx[r[1]], float(r[2]), float(r[3]), float(r[4])) for r in rows], EDGE_DTYPE)
        n50_rows = [(ln.split("\t")[0], int(ln.split("\t")[1])) for ln in open(n50f) if ln.strip()]
        for ani, af in cuts:
            want = replay.greedy_information(tsv, n50f, ani, af)
            assert select.greedy_information(e, edges, paths, n50_rows, ani, af) == want, (gdir, ani, af)
    # this engine's own result: unrounded doubles on the device vs the 2-decimal text the shim writes
    paths = sorted(genomes7)
    edges, _ = e.triangle(screen=80.0, min_af=15.0)
    names = [p.first_name for p in packed]
    tsv = tmp_path / "edges.tsv"
    tsv.write_text(cli.HEADER + "".join(cli.triangle_rows(paths, names, edges)))
    n50f = tmp_path / "n50.tsv"
    n50f.write_text("".join("%s\t%d\n" % (p.path, p.n50) for p in packed))
    n50_rows = [(p.path, p.n50) for p in packed]
    for ani in (97.0, 98.61, 98.73, 99.02, 99.5):  # cutoffs sitting exactly on printed values of this edge list
        for af in (50.0, 89.5, 95.04):
            want = replay.greedy_information(str(tsv), str(n50f), ani, af)
            assert select.greedy_information(e, None, paths, n50_rows, ani, af) == want, (ani, af)  # None: device-resident list
            assert select.greedy_information(e, edges, paths, n50_rows, ani, af) == want, (ani, af)


def test_reference_sharded_triangle_single_process(eng7, ora7, oracle, genomes7, built_lib):
    """The two-step triangle of the multi-GPU path on one device: contexts that own disjoint id ranges of the same
    replicated sketch set, each evaluating the pairs whose reference it owns, together reproduce the full triangle."""
    import ctypes as C

    from skder_b200 import engine

    e, packed = eng7
    full, _ = e.triangle(screen=80.0, min_af=15.0)
    for splits in ([(0, 3), (3, 4)], [(0, 1), (1, 2), (3, 4)]):
        got = []
        for first, count in splits:
            with engine.Engine(0) as e2:
                e2.add(packed)
                e2.index()  # repeat flags of every genome, as the owning rank would have computed them
                e2.set_owned(first, count)
                e2.index()
                ptr, n, st = e2.screen_triangle(80.0)
                assert n == 21 and st.n_pairs_screened == 21
                edges, st2 = e2.pairs_edges(ptr, n, owned_only=True, min_af=15.0)
                assert st2.n_pairs_screened == len(edges)  # every owned pair of this set becomes an edge
                got.append(edges)
                # a pair whose reference lives elsewhere is refused, not answered from a missing table
                sizes = [e2.sizes(g)["n_seeds"] for g in range(7)]
                other = [g for g in range(7) if not (first <= g < first + count)]
                own = [g for g in range(7) if first <= g < first + count]
                bad = [(a, b) for a in own for b in other if sizes[b] > sizes[a]]
                if bad:
                    with pytest.raises(engine.SkbError):
                        e2.pairs_detail([bad[0][0]], [bad[0][1]])
        cat = np.sort(np.concatenate(got), order=["a", "b"])
        covered = sum(c for _, c in splits)
        if covered == 7:
            assert np.array_equal(cat, np.sort(full, order=["a", "b"]))
        else:  # genome 2 is owned by nobody: exactly the pairs with reference 2 are missing
            assert len(cat) < len(full) and set(map(tuple, cat[["a", "b"]].tolist())) < set(map(tuple, full[["a", "b"]].tolist()))


def _bench_line(argv, nproc=1, timeout=900, env=None):
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py")] + argv
    if nproc > 1:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=%d" % nproc, "--master-addr", "127.0.0.1",
               "--master-port", str(29900 + os.getpid() % 90), os.path.join(root, "bench.py")] + argv
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=dict(os.environ, **(env or {})))
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert out.returncode == 0 and lines, out.stdout[-1500:] + out.stderr[-3000:]
    return json.loads(lines[-1])


def test_search_loop_selects_what_the_oracle_loop_selects(built_lib, oracle):
    """bench.py's config4 path (the low_mem_greedy loop of reference skder.py:116-133 on a resident database) on a small
    set of the same shape: as many representatives as the same loop over the oracle's `search`."""
    sys_path = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    import sys

    sys.path.insert(0, sys_path)
    import bench

    want = bench.cpu_search_loop("tiny4", 4, 4, 6)
    got = _bench_line(["--workload", "tiny4", "--steps", "1", "--warmup", "0"])
    assert got["config"]["representatives"] == want["reps"] and got["config"]["pairs"] == want["reps"] * want["n"]
    assert got["config"]["reps_sha256"] == want["reps_sha256"]  # the same genomes, not just as many
    assert got["gpu_launches"] > 0
    # the batched (speculative) loop and the strictly sequential one select the same representatives
    seq = _bench_line(["--workload", "tiny4", "--steps", "1", "--warmup", "0"], env={"SKB_SEARCH_BATCH": "1"})
    assert seq["config"]["reps_sha256"] == got["config"]["reps_sha256"]
