"""`skani`-compatible command line in front of the B200 engine.

skDER reaches its all-vs-all step only through `subprocess.call('skani ...', shell=True)`
(reference src/skDER/util.py:636-652); putting skder_b200/bin/skani first on PATH swaps the engine
without touching skDER.  Sub-commands and flags are exactly the ones skDER spells:

  skani triangle -l LIST --min-af A -E [-s S] -t T -o OUT        (src/skDER/skder.py:16-18,23-25)
  skani sketch   -l LIST -o DBDIR -t T                           (skder.py:103)
  skani search   QUERY.fa -d DBDIR -o OUT -t T                   (skder.py:119)
  skani dist     --rl REFS --ql QUERIES [-s S] [-t T] -o OUT     (skder.py:58-59, cidder.py:362-363)

skani's own command forms work too (DESIGN.md section 3):

  skani triangle [FASTA ...] [-l LIST] -E [-o OUT]       genomes: both sources, deduplicated and sorted
  skani sketch   [FASTA ...] [-l LIST] -o DBDIR          genomes: the FASTAs in order, then the list; nothing deduplicated
  skani dist     [-q FASTA ...] [--ql LIST] [-r FASTA ...] [--rl LIST] [-o OUT]
  skani dist     QUERY REF [REF ...] [-o OUT]
  skani search   QUERY ... [--ql LIST] -d DBDIR [-o OUT]

`-q` / `-r` (dist only) take every following argument up to the next one starting with '-'; each side is its values,
then its list's entries, a path twice on one side counting once.  The positional dist form takes no -q, -r, --ql or
--rl.  Without -o, triangle, dist and search write the TSV to stdout -- the bytes the -o file would hold, nothing on
failure -- and the provenance note below goes to stderr.

`search` also takes several query FASTAs, as positionals and/or a list file `--ql` (positionals first, then the list in
file order, a repeated path once at its first position), answered in one device pass; rows are grouped by query in that
order.  `-n N` (dist, search) keeps each query's first N rows -- its N best hits by unrounded ANI, ties to the reference
listed first; `-n 1` asks for each query's best hit (DESIGN.md section 3).

skDER hands its `-p` string to skani verbatim, so four ANI flags are accepted on triangle, dist and search
(DESIGN.md section 3): the estimators `--median` (median chain identity) and `--robust` (mean after trimming the
10 % / 90 % tails); `--ci`, which appends a bootstrap interval of the mean ANI as two columns, ANI_5_percentile and
ANI_95_percentile; and `--detailed`, which appends 13 columns (contig counts and N90/N50/N10 of both genomes, that
interval, the spread of the chain identities, the chains' average length and the query bases they cover).  --ci and
--detailed are not taken with --median / --robust.  skDER's `-n` clustering reads exactly seven fields (skder.py:190),
so a `-p` with --ci or --detailed breaks it as it would with skani; greedy and dynamic selection are unaffected.
`-m M` (triangle, dist, sketch) is skani's marker compression: a canonical 21-mer is a marker iff its hash is below
2^64 / M (default 1000).  Markers only decide which pairs the prescreen passes, so a smaller M (skani suggests
~200-300 for plasmids and viruses) lets small genomes that share no marker at 1000 be compared; a pair's ANI/AF does
not depend on it.  A database records its M, and `search` sketches the query at that M, so search takes no -m.
skani's per-sequence mode -- `-i` (triangle, sketch), `--qi` (dist, search), `--ri` (dist) -- makes every record of at
least 500 bp of the flagged files a genome of its own, named by its file and header (DESIGN.md section 3); skDER keys
its selection on whole files, so a `-p` with -i breaks it.
Any other skani option (-c, --fast, --slow, --medium, --small-genomes, --no-learned-ani, ...) changes skani's
estimator in ways this engine does not implement: the shim then exits non-zero WITHOUT creating the output, which is
the one failure signal runCmd checks (util.py:642-645).
stderr is discarded by skDER, so diagnostics also go to <output>.skani_b200.log.
"""
import json
import os
import re
import sys
import time

HEADER = "Ref_file\tQuery_file\tANI\tAlign_fraction_ref\tAlign_fraction_query\tRef_name\tQuery_name\n"
# --detailed's columns after the seven above (DESIGN.md section 3); Ref = the edge's genome a, Query = its genome b
DETAILED_COLUMNS = ("Num_ref_contigs", "Num_query_contigs", "ANI_5_percentile", "ANI_95_percentile", "Standard_deviation",
                    "Ref_90_ctg_len", "Ref_50_ctg_len", "Ref_10_ctg_len", "Query_90_ctg_len", "Query_50_ctg_len",
                    "Query_10_ctg_len", "Avg_chain_len", "Total_bases_covered")
DETAILED_FMT = "\t%d\t%d\t%.2f\t%.2f\t%.2f\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\n"
DEFAULT_SCREEN = 80.0  # skani -s default
DEFAULT_MIN_AF = 15.0  # skani --min-af default
DEFAULT_MARKER_C = 1000  # skani -m default


class UsageError(Exception):
    pass


def parse_args(argv):
    """Minimal, strict parser for the skani spellings above.  Returns (subcommand, options dict)."""
    if not argv:
        raise UsageError("no sub-command")
    sub = argv[0]
    if sub not in ("triangle", "sketch", "search", "dist"):
        raise UsageError("unsupported sub-command %r" % sub)
    opt = {"screen": DEFAULT_SCREEN, "min_af": DEFAULT_MIN_AF, "threads": 3, "edge_list": False, "positional": []}
    valued = {
        "-l": "list", "-o": "out", "-t": "threads", "-s": "screen", "--min-af": "min_af", "--rl": "rl", "--ql": "ql",
        "-d": "db", "-m": "marker_c", "-n": "max_results",
    }
    multi = {"-q": "q", "-r": "r"}  # dist's FASTA lists: every following token up to the next one starting with '-'
    flags = {"-E": "edge_list", "--sparse": "edge_list", "--ci": "ci", "--detailed": "detailed", "-i": "per_seq",
             "--qi": "query_per_seq", "--ri": "ref_per_seq"}
    opt["ci"] = opt["detailed"] = opt["per_seq"] = opt["query_per_seq"] = opt["ref_per_seq"] = False
    estimators = {"--median": "median", "--robust": "robust"}
    chosen = []
    i = 1
    while i < len(argv):
        a = argv[i]
        if a == "":
            i += 1
            continue
        if a in valued:
            if i + 1 >= len(argv):
                raise UsageError("option %s needs a value" % a)
            opt[valued[a]] = argv[i + 1]
            i += 2
        elif a in multi:
            vals = opt.setdefault(multi[a], [])
            n0, i = len(vals), i + 1
            while i < len(argv) and not argv[i].startswith("-"):
                if argv[i]:
                    vals.append(argv[i])
                i += 1
            if len(vals) == n0:
                raise UsageError("option %s needs at least one FASTA" % a)
        elif a in flags:
            opt[flags[a]] = True
            i += 1
        elif a in estimators:
            chosen.append(a)
            i += 1
        elif a.startswith("-"):
            raise UsageError("skani option %r is not implemented by the B200 engine" % a)
        else:
            opt["positional"].append(a)
            i += 1
    try:
        opt["screen"] = float(opt["screen"])
        opt["min_af"] = float(opt["min_af"])
        opt["threads"] = max(1, int(opt["threads"]))
    except ValueError as e:
        raise UsageError("bad numeric option: %s" % e)
    if "marker_c" in opt:
        if sub == "search":
            raise UsageError("skani search takes no -m: the query is sketched at the database's marker compression")
        m = opt["marker_c"]
        if not re.fullmatch(r"[0-9]+", m) or not 1 <= int(m) < 2 ** 63:
            raise UsageError("-m needs an integer of at least 1, not %r" % m)
        opt["marker_c"] = int(m)
    else:
        opt["marker_c"] = DEFAULT_MARKER_C
    if "max_results" in opt:
        if sub not in ("search", "dist"):
            raise UsageError("skani %s takes no -n: it is the number of results per query of dist and search" % sub)
        n = opt["max_results"]
        if not re.fullmatch(r"[0-9]+", n) or not 1 <= int(n) < 2 ** 63:
            raise UsageError("-n needs an integer of at least 1, not %r" % n)
        opt["max_results"] = int(n)
    else:
        opt["max_results"] = 0  # every row
    if len(set(chosen)) > 1:
        raise UsageError("--median and --robust are mutually exclusive")
    if chosen and sub == "sketch":
        raise UsageError("skani sketch takes no ANI estimator option (%s)" % chosen[0])
    opt["estimator"] = estimators[chosen[0]] if chosen else "mean"
    if opt["ci"] and sub == "sketch":
        raise UsageError("skani sketch takes no --ci")
    if opt["ci"] and chosen:
        raise UsageError("--ci is defined for the default (mean) ANI only, not with %s" % chosen[0])
    if opt["detailed"] and sub == "sketch":
        raise UsageError("skani sketch takes no --detailed")
    if opt["detailed"] and chosen:
        raise UsageError("--detailed is defined for the default (mean) ANI only, not with %s" % chosen[0])
    for flag, key, subs in (("-i", "per_seq", ("triangle", "sketch")), ("--qi", "query_per_seq", ("dist", "search")),
                            ("--ri", "ref_per_seq", ("dist",))):
        if opt[key] and sub not in subs:
            raise UsageError("skani %s takes no %s (per-sequence mode: %s)" % (sub, flag, ", ".join(subs)))
    if sub != "dist" and ("q" in opt or "r" in opt):
        raise UsageError("skani %s takes no -q / -r: they name dist's query and reference FASTAs" % sub)
    # without -o, triangle, dist and search write the TSV to stdout; sketch writes a directory
    need = {"sketch": ["out"], "search": ["db"]}.get(sub, [])
    for k in need:
        if k not in opt:
            raise UsageError("skani %s: missing required option for %r" % (sub, k))
    if sub in ("triangle", "sketch") and "list" not in opt and not opt["positional"]:
        raise UsageError("skani %s: no genome given (FASTA arguments and/or -l LIST)" % sub)
    if sub == "triangle" and not opt["edge_list"]:
        raise UsageError("skani triangle without -E (matrix output) is not implemented; skDER always passes -E")
    if sub == "search" and not opt["positional"] and "ql" not in opt:
        raise UsageError("skani search: no query FASTA given")
    if sub == "dist":
        lists = [a for a, k in (("-q", "q"), ("-r", "r"), ("--ql", "ql"), ("--rl", "rl")) if k in opt]
        if opt["positional"] and lists:
            raise UsageError("skani dist QUERY REF...: positional FASTAs %r do not combine with %s"
                             % (opt["positional"], ", ".join(lists)))
        if opt["positional"] and len(opt["positional"]) < 2:
            raise UsageError("skani dist QUERY REF [REF ...] needs a query and at least one reference")
        for side, keys in (("query", ("q", "ql")), ("reference", ("r", "rl"))):
            if not opt["positional"] and not any(k in opt for k in keys):
                raise UsageError("skani dist: no %s FASTA given (-%s and/or --%s)" % (side, keys[0], keys[1]))
    return sub, opt


def read_list(path):
    with open(path) as f:
        return [ln.strip() for ln in f if ln.strip()]


def search_queries(opt):
    """search's query FASTAs as given: the positionals, then the --ql list's entries, each path once at its first
    position"""
    qs = list(dict.fromkeys(opt["positional"] + (read_list(opt["ql"]) if "ql" in opt else [])))
    if not qs:
        raise UsageError("skani search: no query FASTA given")
    return qs


def inputs(sub, opt):
    """The FASTA paths a command names, as given, whatever form named them (DESIGN.md section 3):
    triangle: the FASTA arguments and the -l entries, deduplicated and sorted (the triangle's genome order);
    sketch: the FASTA arguments in order, then the -l entries, nothing deduplicated;
    dist: (refs, queries), each -r / -q's values followed by --rl / --ql's entries, or for `dist Q R1 [R2 ...]` the
    first argument as the query and the rest as references (a path twice on one side counts once, in run_dist);
    search: search_queries()."""
    def entries(values_key, list_key):
        return opt.get(values_key, []) + (read_list(opt[list_key]) if list_key in opt else [])

    if sub == "triangle":
        return sorted(set(entries("positional", "list")))
    if sub == "sketch":
        return entries("positional", "list")
    if sub == "dist":
        if opt["positional"]:
            return opt["positional"][1:], opt["positional"][:1]
        return entries("r", "rl"), entries("q", "ql")
    return search_queries(opt)


def emit(opt, text):
    """The TSV into -o, atomically, or without -o onto stdout, written once as a whole so a failure leaves none of it"""
    if "out" in opt:
        write_atomic(opt["out"], text)
    else:
        to_stdout(text)


def to_stdout(data):
    """data, built whole before any of it is written, onto stdout: bytes as they are, text encoded as write_atomic's
    file would be"""
    sys.stdout.flush()
    with open(sys.stdout.fileno(), "wb" if isinstance(data, bytes) else "w", closefd=False) as f:
        f.write(data)


def header(ci, detailed=False):
    if detailed:  # the --ci interval is two of its columns
        return HEADER[:-1] + "".join("\t" + c for c in DETAILED_COLUMNS) + "\n"
    return HEADER[:-1] + "\tANI_5_percentile\tANI_95_percentile\n" if ci else HEADER


def fmt_row(ref, query, ani, af_ref, af_query, ref_name, query_name, ci=None, detail=None):
    row = "%s\t%s\t%.2f\t%.2f\t%.2f\t%s\t%s" % (ref, query, ani, af_ref, af_query, ref_name, query_name)
    if detail is not None:
        return row + DETAILED_FMT % detail
    return row + ("\n" if ci is None else "\t%.2f\t%.2f\n" % ci)


def edge_details(edges, det, n_contigs, nx):
    """--detailed's 13 values per edge, in DETAILED_COLUMNS order.  det: Engine.last_edge_detail() of `edges`;
    n_contigs, nx: Engine.contig_stats() of every genome id the edges hold."""
    nc, nx = n_contigs.tolist(), nx.tolist()
    cols = [edges["a"].tolist(), edges["b"].tolist()]
    cols += [det[k].tolist() for k in ("ani_lo", "ani_hi", "sd", "covered_b", "n_chains")]
    return [(nc[a], nc[b], lo, hi, sd, *nx[a], *nx[b], cov // k, cov) for a, b, lo, hi, sd, cov, k in zip(*cols)]


def write_atomic(path, text):
    d = os.path.dirname(os.path.abspath(path))
    tmp = os.path.join(d, ".%s.tmp.%d" % (os.path.basename(path), os.getpid()))
    with open(tmp, "w") as f:
        f.write(text)
    os.replace(tmp, path)


def _cols(edges, ci, detail):
    """the edges' columns (element access on structured arrays is slow), plus (lo, hi) per edge or None without --ci,
    plus edge_details() per edge or None without --detailed"""
    cols = [edges[k].tolist() for k in ("a", "b", "ani", "af_a", "af_b")]
    cols.append([tuple(x) for x in ci.tolist()] if ci is not None else [None] * len(edges))
    return cols + [detail if detail is not None else [None] * len(edges)]


def triangle_rows(paths_sorted, names, edges, ci=None, detail=None):
    """edges: structured array (a < b, ids index paths_sorted).  Ref = lexicographically smaller path
    (SURVEY.md section 4 fact 3); rows grouped by Ref.  ci: Engine.last_edge_ci() for --ci's two extra columns;
    detail: edge_details() for --detailed's 13 (they replace ci's)."""
    return [fmt_row(paths_sorted[a], paths_sorted[b], ani, afa, afb, names[a], names[b], iv, dt)
            for a, b, ani, afa, afb, iv, dt in zip(*_cols(edges, ci, detail))]


def rect_rows(paths, names, edges, ci=None, detail=None):
    """edges: a = reference id, b = query id.  Rows grouped by query, ANI descending (SURVEY.md section 4 fact 7)."""
    rows = sorted(zip(*_cols(edges, ci, detail)), key=lambda t: (t[1], -t[2], t[0]))
    return [fmt_row(paths[a], paths[b], ani, afa, afb, names[a], names[b], iv, dt)
            for a, b, ani, afa, afb, iv, dt in rows]


def edge_extras(eng, ci, detailed, edges, stats=None):
    """(ci, detail) for triangle_rows / rect_rows after an edge call run with --ci / --detailed as given: stats =
    (n_contigs, nx) of the edges' genome ids, by default Engine.contig_stats of the whole context"""
    if detailed:
        return None, edge_details(edges, eng.last_edge_detail(), *(stats or eng.contig_stats(0, eng.n_genomes)))
    return (eng.last_edge_ci() if ci else None), None


def _device():
    return int(os.environ.get("SKB_DEVICE", os.environ.get("LOCAL_RANK", "0")))


INGEST_BATCH = 256  # genomes packed per host batch: batch k+1 is parsed while batch k uploads and is sketched


def stream_add(eng, engine_mod, paths, threads, phases=None, per_sequence=False):
    """FASTA files -> sketches on the device, streamed: host threads parse and 2-bit pack batch k+1
    (skb_pack_fasta_many) while the device uploads and sketches batch k (skb_add_genomes), so at most two batches of
    packed genomes are resident on the host and the ingest hides behind the upload.  Returns the first-record names.
    per_sequence (-i, --qi, --ri): every kept record is a genome (skb_add_sequences); returns the (file path, record
    name) lists of the genomes added, in id order."""
    from concurrent.futures import ThreadPoolExecutor

    names, gpaths, t_wait, t_add = [], [], 0.0, 0.0
    mcl = eng.params.min_contig_len
    with ThreadPoolExecutor(1) as ex:
        fut = ex.submit(engine_mod.pack_fasta_many, paths[:INGEST_BATCH], threads, mcl) if paths else None
        for i in range(0, len(paths), INGEST_BATCH):
            t0 = time.time()
            packed = fut.result()
            nxt = paths[i + INGEST_BATCH:i + 2 * INGEST_BATCH]
            fut = ex.submit(engine_mod.pack_fasta_many, nxt, threads, mcl) if nxt else None
            t1 = time.time()
            if per_sequence:
                for p in packed:
                    gpaths += [p.path] * p.n_contigs
                    names += p.contig_names
            else:
                names += [p.first_name for p in packed]
            eng.add(packed, per_sequence)
            del packed
            t_wait += t1 - t0
            t_add += time.time() - t1
    if phases is not None:
        phases["ingest_wait_s"] = t_wait  # time the device side waited for the parser (first batch + any shortfall)
        phases["upload_sketch_s"] = t_add
    return (gpaths, names) if per_sequence else names


def _phase_log(opt, phases):
    if os.environ.get("SKB_PHASE_LOG") == "1" and "out" in opt:  # nothing to put it beside with stdout output
        write_atomic(opt["out"].rstrip("/") + ".skani_b200.phases.json", json.dumps(phases))


def run_triangle(opt, engine_mod):
    ph, t0 = {}, time.time()
    paths = inputs("triangle", opt)
    with engine_mod.Engine(_device()) as eng:
        ph["context_s"] = time.time() - t0
        eng.set_estimator(opt["estimator"])
        eng.set_ci(opt["ci"])
        eng.set_detailed(opt["detailed"])
        eng.set_marker_compression(opt["marker_c"])
        if opt["per_seq"]:  # genomes: each file's kept records, files in sorted order
            paths, names = stream_add(eng, engine_mod, paths, opt["threads"], ph, per_sequence=True)
        else:
            names = stream_add(eng, engine_mod, paths, opt["threads"], ph)
        t1 = time.time()
        eng.index()
        t2 = time.time()
        edges, st = eng.triangle(screen=opt["screen"], min_af=opt["min_af"])
        ci, detail = edge_extras(eng, opt["ci"], opt["detailed"], edges)
        t3 = time.time()
    emit(opt, header(opt["ci"], opt["detailed"]) + "".join(triangle_rows(paths, names, edges, ci, detail)))
    ph.update({"index_s": t2 - t1, "triangle_s": t3 - t2, "write_tsv_s": time.time() - t3, "total_s": time.time() - t0,
               "genomes": len(paths), "edges": int(len(edges))})
    _phase_log(opt, ph)
    return st


def run_sketch(opt, engine_mod):
    paths = inputs("sketch", opt)
    os.makedirs(opt["out"], exist_ok=True)
    from . import daemon

    daemon.stop_for(opt["out"])  # a server still holding the previous contents of this directory must not answer for the new ones
    with engine_mod.Engine(_device()) as eng:
        eng.set_marker_compression(opt["marker_c"])  # recorded in the database: its searches sketch queries at it
        if opt["per_seq"]:  # the database's genomes are records: paths[i] is genome i's file, names[i] its header
            paths, names = stream_add(eng, engine_mod, paths, opt["threads"], per_sequence=True)
        else:
            names = stream_add(eng, engine_mod, paths, opt["threads"])
        eng.save(opt["out"])
    write_atomic(os.path.join(opt["out"], "manifest.json"), json.dumps({"paths": paths, "names": names}))


def _daemon_search(opt, labels, dev, out):
    """search through the database's resident daemon (started here if none answers), its TSV written to `out`, an
    absolute path; raises if no server answers or the search fails"""
    import subprocess

    from . import daemon

    db = opt["db"]
    # a per-sequence search is an op of its own, which a server predating it refuses as unknown instead of
    # answering it as a whole-file search
    msg = {"op": "search_records" if opt["query_per_seq"] else "search", "screen": opt["screen"], "min_af": opt["min_af"], "estimator": opt["estimator"],
           "ci": opt["ci"], "detailed": opt["detailed"], "out": out}
    if len(labels) == 1 and not opt["query_per_seq"]:  # the single-query message every server version answers
        msg.update(query=os.path.abspath(labels[0]), label=labels[0])
    else:
        msg.update(queries=[os.path.abspath(q) for q in labels], labels=labels)
    if opt["max_results"]:
        msg["max_results"] = opt["max_results"]
    rep = daemon.request(db, dev, msg)
    if rep is not None and rep.get("error") == "unknown op":  # a server from before this op: replace it, once
        daemon.stop_for(db)
        rep = None
    if rep is not None and rep.get("stale"):  # the directory was rewritten under a running server: it has just exited
        deadline = time.time() + 15.0
        while time.time() < deadline and daemon.request(db, dev, {"op": "ping"}, timeout=1.0) is not None:
            time.sleep(0.05)
        rep = None
    if rep is None:
        log = open(os.path.join(db, "skani_b200_daemon.log"), "a")
        subprocess.Popen([sys.executable, "-m", "skder_b200.daemon", db, str(dev)], stdout=log, stderr=log,
                         stdin=subprocess.DEVNULL, start_new_session=True,
                         cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        deadline = time.time() + float(os.environ.get("SKB_DAEMON_START_TIMEOUT", "600"))
        while rep is None and time.time() < deadline:
            time.sleep(0.2)
            if daemon.request(db, dev, {"op": "ping"}, timeout=5.0):
                rep = daemon.request(db, dev, msg)
    if rep is None:
        raise RuntimeError("search daemon did not come up (see %s/skani_b200_daemon.log)" % db)
    if not rep.get("ok"):
        raise RuntimeError("search daemon: %s" % rep.get("error"))


def run_search(opt, engine_mod):
    """`skani search q.fa [q2.fa ...] [--ql LIST] -d DB [-o OUT]` (reference src/skDER/skder.py:119).  Served by the
    database's resident daemon (skder_b200/daemon.py; started here on first use) unless SKB_NO_DAEMON=1, in which case
    the database is loaded, indexed and searched in this process.  All queries go through one Engine.search."""
    labels = inputs("search", opt)  # each query's rows show its path as it was given
    # the server runs in another working directory: every path goes over absolute
    opt = dict(opt, db=os.path.abspath(opt["db"]))
    if "out" in opt:
        opt["out"] = os.path.abspath(opt["out"])
    dev = _device()
    if os.environ.get("SKB_NO_DAEMON") != "1":
        if "out" in opt:
            _daemon_search(opt, labels, dev, opt["out"])
            return None
        # stdout: the server writes into a fresh private (0700) directory, whose file is copied out; the directory goes
        # on failure too.  No protocol change, so any running server version answers, and the copy is plain file I/O
        # that keeps numpy and the engine out of this process.
        import shutil
        import tempfile

        tmp = tempfile.mkdtemp(prefix="skani_b200.search.")
        try:
            out = os.path.join(tmp, "out.tsv")
            _daemon_search(opt, labels, dev, out)
            with open(out, "rb") as f:
                data = f.read()
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
        to_stdout(data)
        return None
    if engine_mod is None:
        from . import engine as engine_mod
    with open(os.path.join(opt["db"], "manifest.json")) as f:
        man = json.load(f)
    paths, names = list(man["paths"]), list(man["names"])
    with engine_mod.Engine(dev) as eng:
        eng.set_estimator(opt["estimator"])
        eng.set_ci(opt["ci"])
        eng.set_detailed(opt["detailed"])
        eng.set_max_results(opt["max_results"])
        eng.load(opt["db"])
        eng.index()
        qp = engine_mod.pack_fasta_many(labels, opt["threads"], eng.params.min_contig_len)
        edges, st = eng.search(qp, screen=opt["screen"], min_af=opt["min_af"], per_sequence=opt["query_per_seq"])
        ci, detail = edge_extras(eng, opt["ci"], opt["detailed"], edges, search_contig_stats(eng) if opt["detailed"] else None)
    qlabels, qnames = query_columns(labels, qp, opt["query_per_seq"])
    emit(opt, header(opt["ci"], opt["detailed"]) + "".join(rect_rows(paths + qlabels, names + qnames, edges, ci, detail)))
    return st


def query_columns(labels, packed, per_sequence):
    """(Query_file, Query_name) of every query genome of a search: one per file, or with --qi one per kept record"""
    if not per_sequence:
        return list(labels), [p.first_name for p in packed]
    return ([lb for lb, p in zip(labels, packed) for _ in range(p.n_contigs)],
            [n for p in packed for n in p.contig_names])


def search_contig_stats(eng, db_stats=None):
    """contig statistics of the database genomes (db_stats, or read from the context) and, last, of the queries the
    previous Engine.search saw: indexed like the ids of that search's edges"""
    import numpy as np

    cnt, nx = db_stats or eng.contig_stats(0, eng.n_genomes)
    qc, qnx = eng.last_query_contig_stats
    return np.concatenate([cnt, qc]), np.concatenate([nx, qnx])


def run_dist(opt, engine_mod):
    """--ri / --qi split that side's files into records: a (file, split) pair is one unit of genomes, so a file split
    on one side only is compared as records against itself as a whole, and one split on both sides shares its ids"""
    import itertools

    refs, queries = inputs("dist", opt)
    units = list(dict.fromkeys([(p, opt["ref_per_seq"]) for p in refs] + [(p, opt["query_per_seq"]) for p in queries]))
    ids, paths, names = {}, [], []
    with engine_mod.Engine(_device()) as eng:
        eng.set_estimator(opt["estimator"])
        eng.set_ci(opt["ci"])
        eng.set_detailed(opt["detailed"])
        eng.set_marker_compression(opt["marker_c"])
        eng.set_max_results(opt["max_results"])
        for split, run in itertools.groupby(units, key=lambda u: u[1]):
            run = [p for p, _ in run]
            if split:
                gp, gn = stream_add(eng, engine_mod, run, opt["threads"], per_sequence=True)
            else:
                gp, gn = run, stream_add(eng, engine_mod, run, opt["threads"])
            for p in gp:
                ids.setdefault((p, split), []).append(len(paths))
                paths.append(p)
            names += gn

        def genome_ids(side, split):
            return [g for p in dict.fromkeys(side) for g in ids.get((p, split), [])]

        eng.index()
        edges, st = eng.rect(genome_ids(refs, opt["ref_per_seq"]), genome_ids(queries, opt["query_per_seq"]),
                             screen=opt["screen"], min_af=opt["min_af"])
        ci, detail = edge_extras(eng, opt["ci"], opt["detailed"], edges)
    emit(opt, header(opt["ci"], opt["detailed"]) + "".join(rect_rows(paths, names, edges, ci, detail)))
    return st


PROVENANCE = ("skani %s: produced by skder_b200 (B200 engine) in %.2f s -- NOT the skani binary: a restatement of the published "
              "skani method (Shaw & Yu 2023) whose ANI/AF agree with skani's on the reference's golden pairs to sd 0.15 pp "
              "ANI / 0.44 pp AF, out of fold (tests/golden/ORACLE_VS_GOLDEN.md); sketches and prescreen decisions are not "
              "pinned against skani\n")


def _provenance(opt, sub, seconds):
    """Say beside the output which estimator wrote it (skDER discards stdout/stderr).  Overwritten, not appended: the
    search output is rewritten thousands of times by the low_mem_greedy loop."""
    text = PROVENANCE % (sub, seconds)
    if opt.get("estimator", "mean") != "mean":
        text += "ANI estimator: --%s (DESIGN.md section 3)\n" % opt["estimator"]
    if opt.get("ci"):
        text += ("--ci: ANI_5_percentile / ANI_95_percentile are a 100-replicate bootstrap of the pair's chains as DESIGN.md "
                 "section 3 defines it; unpinned against skani's own intervals\n")
    if opt.get("marker_c", DEFAULT_MARKER_C) != DEFAULT_MARKER_C:
        text += ("-m %d: markers are the canonical 21-mers whose hash is below 2^64 / %d (skani's default is 1000); they "
                 "decide only which pairs pass the prescreen, not a pair's ANI/AF\n" % (opt["marker_c"], opt["marker_c"]))
    if opt.get("max_results"):
        text += ("-n %d: each query keeps its first %d rows, by unrounded ANI descending, ties to the lower reference "
                 "id (DESIGN.md section 3); unpinned against skani's own -n\n" % (opt["max_results"], opt["max_results"]))
    if opt.get("per_seq") or opt.get("query_per_seq") or opt.get("ref_per_seq"):
        text += ("%s: per-sequence mode, every record of at least 500 bp is a genome of its own (DESIGN.md section 3); "
                 "skani turns its learned ANI debias off in this mode, this engine keeps its debias substitute on -- the "
                 "difference is unpinned against skani\n"
                 % " ".join(f for f, k in (("-i", "per_seq"), ("--qi", "query_per_seq"), ("--ri", "ref_per_seq")) if opt[k]))
    if opt.get("detailed"):
        text += ("--detailed: the 13 extra columns as DESIGN.md section 3 defines them; their names, order and definitions "
                 "are recalled, unpinned against skani's own --detailed output\n")
    if "out" not in opt:  # the TSV went to stdout: there is no file to put the note beside
        sys.stderr.write(text)
        return
    try:
        write_atomic(opt["out"].rstrip("/") + ".skani_b200.log", text)
    except OSError:
        pass


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    out_hint = None
    t0 = time.time()
    try:
        if "-o" in argv[:-1]:
            out_hint = argv[argv.index("-o") + 1]
        sub, opt = parse_args(argv)
        # A `search` the database's daemon answers needs neither numpy nor the CUDA library in THIS process: skDER's
        # low_mem_greedy loop launches one `skani search` per representative (src/skDER/skder.py:116-120), and importing
        # the engine costs ~0.5 s a time against ~0.1 s for the interpreter plus the socket client.
        engine_mod = None
        if not (sub == "search" and os.environ.get("SKB_NO_DAEMON") != "1"):
            from . import engine as engine_mod  # loads libskani_b200.so; raises if missing (no CPU path)

        {"triangle": run_triangle, "sketch": run_sketch, "search": run_search, "dist": run_dist}[sub](opt, engine_mod)
        _provenance(opt, sub, time.time() - t0)
        return 0
    except Exception as e:  # no output file is left behind: skDER's runCmd then raises
        msg = "skani (B200 engine) failed after %.1fs: %s: %s\nargv: %r\n" % (time.time() - t0, type(e).__name__, e, argv)
        sys.stderr.write(msg)
        if out_hint:
            try:
                with open(out_hint.rstrip("/") + ".skani_b200.log", "a") as f:
                    f.write(msg)
            except OSError:
                pass
        return 2


if __name__ == "__main__":
    sys.exit(main())
