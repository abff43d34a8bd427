"""Resident sketch database for `skani search`.

skDER's low_mem_greedy mode launches one `skani search <genome> -d <db>` process per representative
(reference src/skDER/skder.py:116-120) -- thousands of launches, each of which would otherwise create a
CUDA context, read the database from disk, upload it and build its index.  The first `search` against a
database starts this server (one per database directory, per GPU); it keeps the indexed database in HBM
and answers each later search with one sketch + one rectangle (Engine.search), then exits after
SKB_DAEMON_IDLE seconds without requests.  A request names its query FASTAs as "queries" (absolute paths) and
"labels" (the paths its rows show), or a single one as "query" and "label"; every query of a request is answered in
one device pass.  "max_results" is skani's -n (0 or absent: every row).  The op "search_records" is the same request in
skani's per-sequence mode (--qi): every kept record of the query files is a query.  It is an op of its own so that a
server predating it refuses it as unknown rather than answering it as a whole-file search.

Trust and staleness:
* The Unix socket lives in a directory only the user can enter (mode 0700, ownership checked: $XDG_RUNTIME_DIR
  or /tmp/skb-<uid>), and every connection is authenticated (HMAC challenge of multiprocessing.connection)
  with a random key stored mode 0600 INSIDE the database directory -- whoever can read the database can use its
  server, nobody else, and removing the directory ends the association.  Messages are JSON bytes, never pickles.
* The server remembers the identity (inode, size, mtime) of sketches.skb and manifest.json it loaded and checks it
  before every answer: a database that was rewritten (`skani sketch` into the same directory, as a re-run of
  `skder -d low_mem_greedy` does) is never served from the old copy -- the server says so and exits, the shim starts
  a new one.  `skani sketch` also stops a running server before it writes (stop_for).
"""
import glob
import hashlib
import json
import os
import secrets
import stat
import sys
import time
from multiprocessing.connection import Client, Listener
from multiprocessing import AuthenticationError

IDLE_SECONDS = float(os.environ.get("SKB_DAEMON_IDLE", "900"))


def _runtime_dir():
    base = os.environ.get("SKB_DAEMON_DIR") or os.environ.get("XDG_RUNTIME_DIR")
    d = os.path.join(base, "skb") if base and os.path.isdir(base) else "/tmp/skb-%d" % os.getuid()
    os.makedirs(d, mode=0o700, exist_ok=True)
    st = os.lstat(d)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or (st.st_mode & 0o077):
        raise RuntimeError("socket directory %s is not a private directory of this user" % d)
    return d


def socket_path(db_dir, device):
    key = hashlib.sha256(("%s|%d" % (os.path.realpath(db_dir), device)).encode()).hexdigest()[:24]
    return os.path.join(_runtime_dir(), "%s.sock" % key)


def _key_path(db_dir, device):
    return os.path.join(db_dir, ".skb_daemon.%d.key" % device)


def _read_key(db_dir, device):
    try:
        with open(_key_path(db_dir, device), "rb") as f:
            k = f.read()
        return k if len(k) >= 16 else None
    except OSError:
        return None


def _db_identity(db_dir):
    out = []
    for name in ("sketches.skb", "manifest.json"):
        st = os.stat(os.path.join(db_dir, name))
        out.append((st.st_ino, st.st_size, st.st_mtime_ns))
    return out


def request(db_dir, device, msg, timeout=None):
    """Send one request; returns the reply dict or None if no server of this database is listening."""
    db_dir = os.path.abspath(db_dir)
    key = _read_key(db_dir, device)
    if key is None:
        return None
    try:
        path = socket_path(db_dir, device)
    except RuntimeError:
        return None
    if not os.path.exists(path):
        return None
    try:
        with Client(path, family="AF_UNIX", authkey=key) as conn:
            conn.send_bytes(json.dumps(msg).encode())
            if timeout is not None and not conn.poll(timeout):
                return None
            return json.loads(conn.recv_bytes().decode())
    except (ConnectionRefusedError, FileNotFoundError, EOFError, OSError, AuthenticationError, ValueError):
        return None


def stop_for(db_dir, wait=15.0):
    """Stop every server (any GPU) of this database directory and wait until it is gone."""
    db_dir = os.path.abspath(db_dir)
    for kp in glob.glob(os.path.join(db_dir, ".skb_daemon.*.key")):
        try:
            device = int(os.path.basename(kp).split(".")[2])
        except (IndexError, ValueError):
            continue
        if request(db_dir, device, {"op": "stop"}, timeout=5.0):
            deadline = time.time() + wait
            while time.time() < deadline and os.path.exists(socket_path(db_dir, device)):
                time.sleep(0.05)
        try:
            os.unlink(kp)
        except OSError:
            pass


def search_queries(msg):
    """(query paths, row labels) of a search request: its "queries" / "labels" lists, or its single "query" / "label"
    (the label defaults to the path)"""
    if "queries" in msg:
        queries, labels = list(msg["queries"]), list(msg.get("labels", msg["queries"]))
    else:
        queries, labels = [msg["query"]], [msg.get("label", msg["query"])]
    if not queries or len(labels) != len(queries):
        raise ValueError("a search request needs at least one query and one label per query")
    return queries, labels


def serve(db_dir, device):
    from . import cli, engine

    db_dir = os.path.abspath(db_dir)
    path = socket_path(db_dir, device)
    if os.path.exists(path):
        if request(db_dir, device, {"op": "ping"}, timeout=2.0):
            return 0  # somebody else already serves this database
        os.unlink(path)
    ident = _db_identity(db_dir)
    with open(os.path.join(db_dir, "manifest.json")) as f:
        man = json.load(f)
    paths, names = list(man["paths"]), list(man["names"])
    eng = engine.Engine(device)
    eng.load(db_dir)
    eng.index()
    n_db = eng.n_genomes
    db_stats = None  # contig statistics of the database genomes, read on the first --detailed request
    key = secrets.token_bytes(32)
    kp = _key_path(db_dir, device)
    fd = os.open(kp + ".tmp", os.O_WRONLY | os.O_CREAT | os.O_TRUNC, 0o600)
    with os.fdopen(fd, "wb") as f:
        f.write(key)
    os.replace(kp + ".tmp", kp)
    listener = Listener(path, family="AF_UNIX", authkey=key)
    os.chmod(path, 0o600)
    listener._listener._socket.settimeout(1.0)
    last = time.time()
    try:
        while time.time() - last < IDLE_SECONDS:
            try:
                conn = listener.accept()
            except (TimeoutError, OSError, AuthenticationError, EOFError):
                continue
            stop = False
            with conn:
                try:
                    msg = json.loads(conn.recv_bytes().decode())
                    try:
                        stale = _db_identity(db_dir) != ident
                    except OSError:
                        stale = True
                    if stale and msg.get("op") != "stop":
                        conn.send_bytes(json.dumps({"ok": False, "stale": True, "error": "database directory changed"}).encode())
                        stop = True
                    elif msg.get("op") == "ping":
                        conn.send_bytes(json.dumps({"ok": True, "n": n_db}).encode())
                    elif msg.get("op") == "stop":
                        conn.send_bytes(json.dumps({"ok": True}).encode())
                        stop = True
                    elif msg.get("op") in ("search", "search_records"):
                        per_seq = msg["op"] == "search_records"
                        eng.set_estimator(msg.get("estimator", "mean"))  # per request: a resident server serves every mode
                        ci, detailed = bool(msg.get("ci", False)), bool(msg.get("detailed", False))
                        eng.set_ci(ci)
                        eng.set_detailed(detailed)
                        eng.set_max_results(int(msg.get("max_results", 0)))
                        queries, labels = search_queries(msg)
                        packed = engine.pack_fasta_many(queries, None, eng.params.min_contig_len)
                        edges, st = eng.search(packed, screen=msg["screen"], min_af=msg["min_af"], per_sequence=per_seq)
                        stats = None
                        if detailed:
                            db_stats = db_stats or eng.contig_stats(0, n_db)  # the database's, once per server
                            stats = cli.search_contig_stats(eng, db_stats)
                        qlabels, qnames = cli.query_columns(labels, packed, per_seq)
                        rows = cli.rect_rows(paths + qlabels, names + qnames, edges,
                                             *cli.edge_extras(eng, ci, detailed, edges, stats))
                        cli.write_atomic(msg["out"], cli.header(ci, detailed) + "".join(rows))
                        conn.send_bytes(json.dumps({"ok": True, "rows": len(rows), "ms": st.ms_total}).encode())
                    else:
                        conn.send_bytes(json.dumps({"ok": False, "error": "unknown op"}).encode())
                except Exception as e:  # the shim turns this into "no output file"
                    try:
                        conn.send_bytes(json.dumps({"ok": False, "error": "%s: %s" % (type(e).__name__, e)}).encode())
                    except Exception:
                        pass
            if stop:
                break
            last = time.time()
    finally:
        listener.close()
        if os.path.exists(path):
            os.unlink(path)
        if _read_key(db_dir, device) == key:
            try:
                os.unlink(kp)
            except OSError:
                pass
        eng.close()
    return 0


if __name__ == "__main__":
    sys.exit(serve(sys.argv[1], int(sys.argv[2]) if len(sys.argv) > 2 else 0))
