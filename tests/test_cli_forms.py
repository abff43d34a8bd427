"""skani's own command forms (DESIGN.md section 3): FASTA arguments on triangle and sketch, -q / -r and `dist Q R...` on
dist, and the TSV on stdout without -o.  The parser's resolved inputs and refusals; the CPU reference
(tests/cli_forms_ref.py) against hand-written list-file commands through the oracle; stdout on failure and through a
stand-in search server; and on the device every new form byte-identical to its list-file form and to the reference."""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 20261024
SHIM = os.path.join(ROOT, "skder_b200", "bin", "skani")
REF = os.path.join(ROOT, "tests", "cli_forms_ref.py")
LIST_REF = os.path.join(ROOT, "tests", "per_sequence_ref.py")


def _run(script, argv, env=None, cwd=None):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, script] + argv, capture_output=True, env=e, cwd=cwd, timeout=900)


def _output(script, argv, env=None):
    """what a command wrote: its -o file, or without -o its stdout (bytes); asserts exit 0"""
    if "-o" in argv:
        out = argv[argv.index("-o") + 1]
        if os.path.exists(out):
            os.unlink(out)
    r = _run(script, argv, env)
    assert r.returncode == 0, (argv, r.stderr.decode())
    if "-o" not in argv:
        return r.stdout
    assert r.stdout == b"", argv
    with open(out, "rb") as f:
        return f.read()


def _lst(path, items):
    path.write_text("".join(x + "\n" for x in items))
    return str(path)


# ---- the parser ---------------------------------------------------------------------------------------------------------
def test_inputs_of_every_form(tmp_path):
    from skder_b200 import cli

    L = _lst(tmp_path / "l.txt", ["c.fa", "a.fa", "c.fa"])
    QL = _lst(tmp_path / "ql.txt", ["q3.fa", "q1.fa"])
    RL = _lst(tmp_path / "rl.txt", ["r2.fa"])

    def inputs(*argv):
        sub, opt = cli.parse_args(list(argv))
        return cli.inputs(sub, opt)

    # triangle: both sources, deduplicated and sorted; -i applies whichever way a genome came
    assert inputs("triangle", "b.fa", "a.fa", "b.fa", "-E") == ["a.fa", "b.fa"]
    assert inputs("triangle", "-l", L, "-E", "-o", "o") == ["a.fa", "c.fa"]
    assert inputs("triangle", "d.fa", "-l", L, "b.fa", "", "-E") == ["a.fa", "b.fa", "c.fa", "d.fa"]
    _, opt = cli.parse_args(["triangle", "b.fa", "a.fa", "-E", "-i"])
    assert opt["per_seq"] and "out" not in opt
    # sketch: FASTA arguments in order, then the list, duplicates kept
    assert inputs("sketch", "b.fa", "a.fa", "a.fa", "-o", "db") == ["b.fa", "a.fa", "a.fa"]
    assert inputs("sketch", "b.fa", "-l", L, "-o", "db", "a.fa") == ["b.fa", "a.fa", "c.fa", "a.fa", "c.fa"]
    assert inputs("sketch", "-l", L, "-o", "db") == ["c.fa", "a.fa", "c.fa"]
    # dist, list form: (refs, queries), values first, then the list's entries
    assert inputs("dist", "--rl", RL, "--ql", QL, "-o", "o") == (["r2.fa"], ["q3.fa", "q1.fa"])
    assert inputs("dist", "-q", "q1.fa", "q2.fa", "-r", "r1.fa") == (["r1.fa"], ["q1.fa", "q2.fa"])
    assert inputs("dist", "--ql", QL, "-r", "r1.fa", "r3.fa", "-q", "q9.fa", "--rl", RL, "-n", "2") == \
        (["r1.fa", "r3.fa", "r2.fa"], ["q9.fa", "q3.fa", "q1.fa"])
    assert inputs("dist", "-q", "a.fa", "", "b.fa", "-r", "c.fa", "", "-o", "o") == (["c.fa"], ["a.fa", "b.fa"])
    assert inputs("dist", "-q", "a.fa", "-q", "b.fa", "-r", "c.fa", "c.fa") == (["c.fa", "c.fa"], ["a.fa", "b.fa"])
    _, opt = cli.parse_args(["dist", "-q", "a.fa", "-r", "c.fa", "--qi", "--ri", "-o", "o"])
    assert opt["query_per_seq"] and opt["ref_per_seq"] and opt["out"] == "o" and opt["q"] == ["a.fa"]
    # dist, positional form: the first is the query, the rest the references
    assert inputs("dist", "q.fa", "r1.fa", "r2.fa") == (["r1.fa", "r2.fa"], ["q.fa"])
    assert inputs("dist", "q.fa", "", "r1.fa", "-s", "85", "--ci") == (["r1.fa"], ["q.fa"])
    # search: unchanged
    assert inputs("search", "b.fa", "-d", "db", "--ql", QL, "b.fa") == ["b.fa", "q3.fa", "q1.fa"]
    _, opt = cli.parse_args(["search", "b.fa", "-d", "db"])
    assert "out" not in opt


def test_refusals():
    from skder_b200 import cli

    bad = [
        # -q / -r off dist
        "triangle -q a.fa -E", "triangle -l L -E -r a.fa", "sketch -q a.fa -o db", "sketch a.fa -r b.fa -o db",
        "search a.fa -d db -q b.fa", "search -d db -r a.fa",
        # positional dist mixed with list options, or a single positional
        "dist a.fa b.fa -q c.fa", "dist a.fa b.fa -r c.fa", "dist a.fa b.fa --rl R", "dist a.fa b.fa --ql Q",
        "dist --rl R --ql Q -o o a.fa", "dist -q a.fa -r b.fa c.fa -o o d.fa -s 85 e.fa", "dist a.fa", "dist a.fa -o o",
        # an empty -q / -r
        "dist -q -r a.fa", "dist -r a.fa -q", "dist -q -o o -r a.fa", "dist -r a.fa -q --ql Q",
        # no genomes, or one side missing
        "triangle -E -o o", "triangle -E", "sketch -o db", "dist -o o", "dist", "dist -q a.fa", "dist -r a.fa --rl R",
        "dist --ql Q", "search -d db", "search -d db -o o",
        # sketch writes a directory: -o stays required
        "sketch a.fa b.fa", "sketch -l L",
        # refusals that stand in every form: matrix output, the sketch / estimator options
        "triangle a.fa b.fa -o o", "triangle a.fa b.fa", "triangle a.fa -E -c 30", "triangle a.fa b.fa -E --fast",
        "dist a.fa b.fa --no-learned-ani", "dist -q a.fa -r b.fa --slow", "sketch a.fa -o db --small-genomes",
        "search a.fa -d db --medium", "dist a.fa b.fa -i", "dist -q a.fa -r b.fa -m 0",
    ]
    for argv in bad:
        with pytest.raises(cli.UsageError):
            cli.parse_args(argv.split())
    with pytest.raises(cli.UsageError):
        cli.parse_args(["dist", "-q", "", "-r", "a.fa"])


def test_refusals_leave_no_output(tmp_path):
    out = tmp_path / "o.tsv"
    cwd = tmp_path / "cwd"
    cwd.mkdir()
    for argv in (["triangle", "a.fa", "b.fa"], ["triangle", "a.fa", "b.fa", "-E", "--fast"],
                 ["dist", "a.fa", "b.fa", "--no-learned-ani"], ["dist", "-q", "a.fa", "-r", "b.fa", "-c", "30"],
                 ["dist", "a.fa", "b.fa", "--rl", "r"], ["search", "a.fa", "-d", "db", "-q", "b.fa"]):
        r = _run(SHIM, argv + ["-o", str(out)], {"SKB_NO_DAEMON": "1"})
        assert r.returncode != 0 and not out.exists() and r.stdout == b"", argv
        r = _run(SHIM, argv, {"SKB_NO_DAEMON": "1"}, cwd=str(cwd))  # the stdout form
        assert r.returncode != 0 and r.stdout == b"" and b"UsageError" in r.stderr, argv
    assert os.listdir(cwd) == []


def test_stdout_failure_writes_nothing(tmp_path):
    """a genome or database that cannot be read: non-zero exit, nothing on stdout, the message on stderr, no file"""
    from skder_b200 import synth

    g = str(tmp_path / "g.fa")
    synth.write_fasta(g, [b"ACGT" * 500])
    missing = str(tmp_path / "missing.fa")
    for argv in (["triangle", g, missing, "-E"], ["dist", g, missing], ["dist", "-q", missing, "-r", g],
                 ["search", g, "-d", str(tmp_path / "no_db")]):
        r = _run(SHIM, argv, {"SKB_NO_DAEMON": "1"}, cwd=str(tmp_path))
        assert r.returncode != 0 and r.stdout == b"", argv
        assert b"skani (B200 engine) failed" in r.stderr, argv
    assert sorted(os.listdir(tmp_path)) == ["g.fa"]


# ---- the CPU reference against hand-written list-file commands ----------------------------------------------------------
def test_reference_equals_list_files(oracle, genomes7, tmp_path):
    G = genomes7
    n = [0]

    def lst(items):
        n[0] += 1
        return _lst(tmp_path / ("l%d.txt" % n[0]), items)

    L = lst([G[0], G[3], G[5]])
    RL, QL = lst([G[4], G[2]]), lst([G[6], G[0]])
    db = str(tmp_path / "db")
    assert _run(os.path.join(ROOT, "tests", "oracle_skani.py"), ["sketch", "-l", lst(G[2:]), "-o", db]).returncode == 0
    f_old, f_new = str(tmp_path / "old.tsv"), str(tmp_path / "new.tsv")
    cases = [
        (["triangle", G[2], G[1], G[3], "-l", L, "-E"], ["triangle", "-l", lst([G[2], G[1], G[3]] + [G[0], G[3], G[5]]), "-E"]),
        (["triangle", *G[3:], "-E", "-s", "85", "--ci"], ["triangle", "-l", lst(G[3:]), "-E", "-s", "85", "--ci"]),
        (["dist", "-q", G[0], G[1], "-r", G[2], "--rl", RL, "-n", "2"],
         ["dist", "--ql", lst([G[0], G[1]]), "--rl", lst([G[2], G[4], G[2]]), "-n", "2"]),
        (["dist", "--ql", QL, "-r", G[1], G[5], "-q", G[3], "--detailed"],
         ["dist", "--ql", lst([G[3], G[6], G[0]]), "--rl", lst([G[1], G[5]]), "--detailed"]),
        (["dist", "-r", G[0], G[0], G[1], "-q", G[2], G[1], G[2], "--median"],
         ["dist", "--rl", lst([G[0], G[0], G[1]]), "--ql", lst([G[2], G[1], G[2]]), "--median"]),
        (["dist", G[6], *G[:4]], ["dist", "--ql", lst([G[6]]), "--rl", lst(G[:4])]),
        (["search", G[0], G[1], "-d", db, "-n", "2"], ["search", G[0], G[1], "-d", db, "-n", "2"]),
    ]
    for new, old in cases:
        want = _output(LIST_REF, old + ["-o", f_old])
        assert want.count(b"\n") > 2, old
        assert _output(REF, new + ["-o", f_new]) == want, new
        assert _output(REF, new) == want, new
    # sketch: the FASTA arguments, then the list, as one -l list
    dbs = [str(tmp_path / d) for d in ("db_new", "db_old")]
    assert _run(REF, ["sketch", G[1], G[0], "-l", L, "-o", dbs[0]]).returncode == 0
    assert _run(LIST_REF, ["sketch", "-l", lst([G[1], G[0], G[0], G[3], G[5]]), "-o", dbs[1]]).returncode == 0
    man = [open(os.path.join(d, "manifest.json")).read() for d in dbs]
    assert man[0] == man[1] and json.loads(man[0])["paths"] == [G[1], G[0], G[0], G[3], G[5]]


# ---- search through a stand-in server -----------------------------------------------------------------------------------
ROWS = "Ref_file\tQuery_file\tANI\tAlign_fraction_ref\tAlign_fraction_query\tRef_name\tQuery_name\n/r.fa\tq1.fa\t99.00" \
       "\t90.00\t91.00\tr é\tq\n".encode()


def _search_through_stand_in(tmp_path, reply):
    """the shim's `search q1.fa -d DB` without -o against a stand-in server that writes ROWS to the path it is given and
    answers `reply`; returns (the finished process, the message, the mode of the directory holding the output path,
    the client's 'numpy imported' / 'engine imported' / exit code as printed on stderr)"""
    from multiprocessing.connection import Listener

    from skder_b200 import daemon

    db = tmp_path / "db"
    db.mkdir(exist_ok=True)
    tmpdir = tmp_path / "tmp"
    tmpdir.mkdir(exist_ok=True)
    run_dir = tempfile.mkdtemp(prefix="skb-", dir="/tmp")  # a Unix socket path holds at most 107 bytes
    env = dict(os.environ, SKB_DAEMON_DIR=run_dir, SKB_DEVICE="0", PYTHONPATH=ROOT, TMPDIR=str(tmpdir))
    env.pop("SKB_NO_DAEMON", None)
    os.environ["SKB_DAEMON_DIR"] = run_dir
    try:
        sock = daemon.socket_path(str(db), 0)
    finally:
        os.environ.pop("SKB_DAEMON_DIR", None)
    key = b"k" * 32
    with open(daemon._key_path(str(db), 0), "wb") as f:
        f.write(key)
    seen = []

    def serve():
        with Listener(sock, family="AF_UNIX", authkey=key) as ls:
            with ls.accept() as conn:
                msg = json.loads(conn.recv_bytes().decode())
                seen.append((msg, os.stat(os.path.dirname(msg["out"])).st_mode & 0o777))
                with open(msg["out"], "wb") as f:
                    f.write(ROWS)
                conn.send_bytes(json.dumps(reply).encode())

    th = threading.Thread(target=serve, daemon=True)
    th.start()
    for _ in range(200):
        if os.path.exists(sock):
            break
        time.sleep(0.01)
    code = ("import sys; from skder_b200.cli import main; rc = main(sys.argv[1:]); "
            "sys.stderr.write('\\nimports: %s %s %d\\n' % ('numpy' in sys.modules, 'skder_b200.engine' in sys.modules, rc)); sys.exit(rc)")
    try:
        r = subprocess.run([sys.executable, "-c", code, "search", "q1.fa", "-d", str(db)], capture_output=True, env=env,
                           cwd=str(tmp_path), timeout=60)
        th.join(timeout=10)
    finally:
        shutil.rmtree(run_dir, ignore_errors=True)
    imports = r.stderr.decode().rsplit("imports: ", 1)[1].split()
    assert os.listdir(tmpdir) == [], "the private output directory is removed"
    return r, seen[0][0], seen[0][1], imports


def test_stdout_search_through_daemon(tmp_path):
    r, msg, mode, imports = _search_through_stand_in(tmp_path, {"ok": True})
    assert r.returncode == 0, r.stderr.decode()
    assert r.stdout == ROWS
    assert imports == ["False", "False", "0"]
    assert mode == 0o700 and os.path.isabs(msg["out"]) and not os.path.exists(os.path.dirname(msg["out"]))
    assert msg["op"] == "search" and msg["query"] == str(tmp_path / "q1.fa") and msg["label"] == "q1.fa"
    assert b"NOT the skani binary" in r.stderr  # the provenance note goes to stderr
    assert sorted(os.listdir(tmp_path)) == ["db", "tmp"]


def test_stdout_search_through_daemon_failure(tmp_path):
    r, msg, _, imports = _search_through_stand_in(tmp_path, {"ok": False, "error": "stand-in refuses"})
    assert r.returncode != 0 and r.stdout == b"" and b"stand-in refuses" in r.stderr
    assert imports == ["False", "False", "2"]
    assert not os.path.exists(os.path.dirname(msg["out"]))


# ---- on the device ------------------------------------------------------------------------------------------------------
def multi_fastas(d):
    """two multi-record files over two clades of 20 kb sequences, with a record under 500 bp, and a one-record file"""
    from skder_b200 import synth

    cl = [[g[0] for g in synth.one_clade(c, 4, 20_000, SEED, d_lo=0.001, d_hi=0.01, max_contigs=1)] for c in range(2)]
    files = {"m1.fa": [cl[0][0], cl[1][0], b"ACGT" * 100, cl[0][1]], "m2.fa": [cl[1][1], cl[0][2], cl[1][2]],
             "m3.fa": [cl[0][3]]}
    paths = []
    for name, recs in files.items():
        paths.append(str(d / name))
        synth.write_fasta(paths[-1], recs, name=name.split(".")[0])
    return paths


def _db_files(d):
    return {f: open(os.path.join(d, f), "rb").read() for f in sorted(os.listdir(d))
            if not f.startswith(".") and not f.startswith("skani_b200_daemon")}


@pytest.mark.gpu
def test_new_forms_equal_list_forms(built_lib, genomes7, tmp_path):
    from skder_b200 import daemon

    G = genomes7
    M = multi_fastas(tmp_path)
    n = [0]

    def lst(items):
        n[0] += 1
        return _lst(tmp_path / ("l%d.txt" % n[0]), items)

    f_old, f_new = str(tmp_path / "old.tsv"), str(tmp_path / "new.tsv")

    def check(new, old, env=None):
        """the list-file form's output; the new form's -o file and stdout and the CPU reference's stdout equal it"""
        want = _output(SHIM, old + ["-o", f_old], env)
        assert want.count(b"\n") > 2, old
        assert _output(SHIM, new + ["-o", f_new], env) == want, new
        assert _output(SHIM, new, env) == want, new
        assert _output(REF, new) == want, new

    L = lst([G[0], G[5], G[2]])
    for extra in ([], ["--ci", "-m", "200"], ["--detailed", "-s", "85", "--min-af", "20"], ["--median"], ["--robust"]):
        check(["triangle", G[6], G[2], "-l", L, G[1], "-E", "-t", "4"] + extra,
              ["triangle", "-l", lst([G[0], G[1], G[2], G[5], G[6]]), "-E", "-t", "4"] + extra)
    for extra in (["-i"], ["-i", "--detailed", "-m", "200"]):
        check(["triangle", *M, "-E"] + extra, ["triangle", "-l", lst(M), "-E"] + extra)
    RL = lst([G[4], G[2]])
    for extra in ([], ["-n", "2"], ["--ci"], ["--robust", "-n", "1"]):
        check(["dist", "-q", G[0], G[1], G[0], "-r", G[2], G[3], "--rl", RL] + extra,
              ["dist", "--ql", lst([G[0], G[1], G[0]]), "--rl", lst([G[2], G[3], G[4], G[2]])] + extra)
    for extra in ([], ["--detailed"], ["--median", "-s", "85"]):
        check(["dist", G[6], *G[:4]] + extra, ["dist", "--ql", lst([G[6]]), "--rl", lst(G[:4])] + extra)
    for extra in (["--qi"], ["--ri", "-m", "200"], ["--qi", "--ri", "-n", "2", "--ci"], ["--qi", "--min-af", "30"]):
        check(["dist", "-q", M[0], "-r", M[1], M[2]] + extra, ["dist", "--ql", lst(M[:1]), "--rl", lst(M[1:])] + extra)
        check(["dist", M[0], M[1], M[2]] + extra, ["dist", "--ql", lst(M[:1]), "--rl", lst(M[1:])] + extra)
    # sketch from FASTA arguments: the same database as from -l, and the same search answers against either
    dbs = {}
    for name, form in (("new", [G[3], G[2], "-l", lst(G[4:])]), ("old", ["-l", lst([G[3], G[2]] + G[4:])]),
                       ("new_i", [*M, "-i", "-m", "200"]), ("old_i", ["-l", lst(M), "-i", "-m", "200"])):
        dbs[name] = str(tmp_path / ("db_" + name))
        r = _run(SHIM, ["sketch"] + form + ["-o", dbs[name]])
        assert r.returncode == 0, r.stderr.decode()
    for a, b in (("new", "old"), ("new_i", "old_i")):
        fa, fb = _db_files(dbs[a]), _db_files(dbs[b])
        assert fa == fb and "manifest.json" in fa and len(fa) > 1, (sorted(fa), sorted(fb))
    QL = lst([G[1]])
    try:
        for env in ({"SKB_NO_DAEMON": "1"}, {"SKB_DAEMON_IDLE": "120"}):
            for db in (dbs["new"], dbs["old"]):
                for extra in ([], ["-n", "2"], ["--detailed"], ["--median"]):
                    check(["search", G[0], "-d", db, "--ql", QL] + extra,
                          ["search", G[0], "-d", dbs["old"], "--ql", QL] + extra, env)
            for extra in (["--qi"], ["--qi", "-n", "1", "--ci"]):
                check(["search", M[1], "-d", dbs["new_i"]] + extra, ["search", M[1], "-d", dbs["old_i"]] + extra, env)
    finally:
        for db in dbs.values():
            daemon.stop_for(db)
