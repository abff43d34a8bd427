"""skani's per-sequence mode (-i, --qi, --ri) on top of the CPU references -- TEST INFRASTRUCTURE ONLY.

`python tests/per_sequence_ref.py <skani argv>` is the CPU `skani` for these flags (DESIGN.md section 3).  Every record
of at least min_contig_len (500) bases of a split file is a genome of its own, sketched by oracle.Sketch.from_contigs
from that record alone.  The run itself is tests/search_queries_ref.py (and through it the -m, estimator, --ci and
--detailed references) over list files that name each record by a key `<path>\\x01<record index, 9 digits>`: keys sort
like (path, record), which is triangle's genome order, and the oracle's Sketch.from_file is pointed at the record for a
key while the run lasts.  The file and name columns of the output are then relabelled to the record's file and header.
The oracle and the other references are unchanged.

A database's manifest names genome i's file as paths[i].  A file that occurs there exactly as often as it has kept
records was sketched with -i (its k-th occurrence is its k-th record); any other occurrence is a whole file.  The two
readings agree for a file with one kept record.
"""
import contextlib
import gzip
import json
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402

MIN_CONTIG_LEN = 500
SEP = "\x01"


def records(path, min_len=MIN_CONTIG_LEN):
    """[(header without '>', sequence)] of the records of at least min_len bases, as the packer keeps them: a '>' at a
    line start opens a record, blanks (space, tab, CR) inside sequence lines are dropped, CRs end a header"""
    with open(path, "rb") as f:
        data = f.read()
    if data[:2] == b"\x1f\x8b":
        data = gzip.decompress(data)
    out, name, seq = [], None, []
    for line in data.split(b"\n"):
        if line.startswith(b">"):
            if name is not None:
                out.append((name, b"".join(seq)))
            name, seq = line[1:].rstrip(b"\r"), []
        elif name is not None:
            seq.append(line.translate(None, b" \t\r"))
    if name is not None:
        out.append((name, b"".join(seq)))
    return [(n.decode("utf-8", "replace"), s) for n, s in out if len(s) >= min_len and len(s) > 0]


def key(path, k):
    return "%s%s%09d" % (path, SEP, k)


class Records:
    """the keys of split files and what each stands for"""

    def __init__(self):
        self.rec = {}  # key -> (path, header, sequence)
        self.cache = {}

    def split(self, path):
        if path not in self.cache:
            self.cache[path] = records(path)
        keys = []
        for k, (name, seq) in enumerate(self.cache[path]):
            keys.append(key(path, k))
            self.rec[keys[-1]] = (path, name, seq)
        return keys

    @contextlib.contextmanager
    def sketches(self):
        """Sketch.from_file of a key sketches its record alone"""
        orig = O.Sketch.__dict__["from_file"]
        rec = self.rec

        def from_file(cls, path, params=None):
            if path in rec:
                return cls.from_contigs([rec[path][2]], params)
            return orig.__func__(cls, path, params)

        O.Sketch.from_file = classmethod(from_file)
        try:
            yield
        finally:
            O.Sketch.from_file = orig

    def relabel(self, text):
        lines = text.splitlines(keepends=True)
        out = [lines[0]]
        for ln in lines[1:]:
            t = ln.rstrip("\n").split("\t")
            for col, name_col in ((0, 5), (1, 6)):
                if t[col] in self.rec:
                    path, name, _ = self.rec[t[col]]
                    t[col], t[name_col] = path, name
            out.append("\t".join(t) + "\n")
        return "".join(out)


def replace(argv, values, drop_flags=(), positionals=None):
    """argv with the valued options in `values` set to the given value (None: dropped) and the flags in drop_flags
    dropped; positionals (a list) replaces search's positional arguments"""
    from search_queries_ref import VALUED

    out, i = [argv[0]], 1
    while i < len(argv):
        a = argv[i]
        if a in VALUED:
            if a not in values:
                out += argv[i:i + 2]
            i += 2
        elif a in drop_flags:
            i += 1
        elif positionals is not None and a and not a.startswith("-"):
            i += 1
        else:
            out.append(a)
            i += 1
    for a, v in values.items():
        if v is not None:
            out += [a, v]
    return out + list(positionals or [])


def main(argv):
    import marker_c_ref
    import search_queries_ref
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)
    if not (opt["per_seq"] or opt["query_per_seq"] or opt["ref_per_seq"] or sub == "search"):
        return search_queries_ref.main(argv)
    R = Records()
    tmp = tempfile.mkdtemp(prefix="per_seq_ref.")
    out = os.path.join(tmp, "out.tsv")
    flags = ("-i", "--qi", "--ri")

    def listfile(name, keys):
        p = os.path.join(tmp, name)
        with open(p, "w") as f:
            f.write("".join(k + "\n" for k in keys))
        return p

    try:
        with R.sketches():
            if sub in ("triangle", "sketch"):
                paths = cli.read_list(opt["list"])
                files = sorted(set(paths)) if sub == "triangle" else list(dict.fromkeys(paths))
                keys = [k for p in files for k in R.split(p)]
                if sub == "sketch":
                    rc = search_queries_ref.main(replace(argv, {"-l": listfile("l.txt", keys)}, flags))
                    if rc == 0:
                        man = os.path.join(opt["out"], "manifest.json")
                        with open(man) as f:
                            d = json.load(f)
                        d.update(paths=[R.rec[k][0] for k in keys], names=[R.rec[k][1] for k in keys])
                        cli.write_atomic(man, json.dumps(d))
                    return rc
                rc = search_queries_ref.main(replace(argv, {"-l": listfile("l.txt", keys), "-o": out}, flags))
            elif sub == "dist":
                def side(paths, split):
                    return [k for p in dict.fromkeys(paths) for k in (R.split(p) if split else [p])]

                rl = side(cli.read_list(opt["rl"]), opt["ref_per_seq"])
                ql = side(cli.read_list(opt["ql"]), opt["query_per_seq"])
                rc = search_queries_ref.main(replace(argv, {"--rl": listfile("rl.txt", rl),
                                                            "--ql": listfile("ql.txt", ql), "-o": out}, flags))
            else:  # search: the database's genomes as keys, then the queries
                with open(os.path.join(opt["db"], "manifest.json")) as f:
                    db_paths = json.load(f)["paths"]
                seen, db_keys = {}, []
                for p in db_paths:
                    k = seen[p] = seen.get(p, -1) + 1
                    db_keys.append(key(p, k) if db_paths.count(p) == len(R.split(p)) else p)
                db = os.path.join(tmp, "db")
                os.makedirs(db)
                with open(os.path.join(db, "manifest.json"), "w") as f:
                    json.dump({"paths": db_keys, "marker_c": marker_c_ref.db_marker_c(opt["db"])}, f)
                queries = cli.search_queries(opt)
                if opt["query_per_seq"]:
                    queries = [k for q in queries for k in R.split(q)]
                rc = search_queries_ref.main(replace(argv, {"-d": db, "--ql": listfile("ql.txt", queries), "-o": out},
                                                     flags, positionals=[]))
        if rc == 0:
            with open(out) as f:
                cli.write_atomic(opt["out"], R.relabel(f.read()))
        return rc
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
