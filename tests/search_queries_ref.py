"""Several queries per `skani search` and skani's -n on search / dist, on top of the CPU references -- TEST
INFRASTRUCTURE ONLY.

`python tests/search_queries_ref.py <skani argv>` is the CPU `skani` for these options: tests/marker_c_ref.py (itself
oracle_skani.py with the estimator, --ci and --detailed references, at the database's or the argv's -m) run once per
search query, the outputs concatenated in query order (DESIGN.md section 3: the positionals, then the --ql list, each
path once).  With -n N every query keeps its first N rows after ordering them by the unrounded ANI of the oracle with
the active estimator, descending, ties to the lower reference id (the reference's position in the database manifest
for search, in the dist id list otherwise); the kept rows stay in the order the reference wrote them.  The references
themselves are unchanged.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# skani options that take a value (skder_b200/cli.py parse_args)
VALUED = ("-l", "-o", "-t", "-s", "--min-af", "--rl", "--ql", "-d", "-m", "-n")


def strip(argv, drop, positionals=False):
    """argv without the valued options in `drop` (and their values) and, if positionals, without positional args"""
    out, i = [argv[0]], 1
    while i < len(argv):
        a = argv[i]
        if a in VALUED:
            if a not in drop:
                out += argv[i:i + 2]
            i += 2
            continue
        if positionals and a and not a.startswith("-"):
            i += 1
            continue
        out.append(a)
        i += 1
    return out


def cut(lines, ref_id, n, mode):
    """the rows (TSV lines, grouped by Query_file) each query keeps under -n n, in their order"""
    import ani_estimators_ref as EST
    from oracle import oracle as O

    sk = {}

    def ani(r, q):
        for p in (r, q):
            if p not in sk:
                sk[p] = O.Sketch.from_file(p)
        return EST.pair(sk[r], sk[q], None, mode).ani

    groups = {}
    for i, ln in enumerate(lines):
        t = ln.split("\t")
        groups.setdefault(t[1], []).append((-ani(t[0], t[1]), ref_id[t[0]], i))
    keep = {i for g in groups.values() for _, _, i in sorted(g)[:n]}
    return [ln for i, ln in enumerate(lines) if i in keep]


def _lines(path):
    with open(path) as f:
        return f.read().splitlines(keepends=True)


def main(argv):
    import marker_c_ref
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)
    n = opt["max_results"]
    if sub == "dist":
        rc = marker_c_ref.main(strip(argv, ("-n",)))
        if rc or not n:
            return rc
        paths = list(dict.fromkeys(cli.read_list(opt["rl"]) + cli.read_list(opt["ql"])))
        lines = _lines(opt["out"])
        body = cut(lines[1:], {p: i for i, p in enumerate(paths)}, n, opt["estimator"])
        cli.write_atomic(opt["out"], lines[0] + "".join(body))
        return 0
    if sub != "search":
        return marker_c_ref.main(argv)
    with open(os.path.join(opt["db"], "manifest.json")) as f:
        ref_id = {p: i for i, p in enumerate(json.load(f)["paths"])}
    base = strip(argv, ("-n", "--ql", "-o"), positionals=True)
    head, body = None, []
    for k, q in enumerate(cli.search_queries(opt)):
        tmp = "%s.query%d.tmp" % (opt["out"], k)
        try:
            rc = marker_c_ref.main(base[:1] + [q] + base[1:] + ["-o", tmp])
            if rc:
                return rc
            lines = _lines(tmp)
        finally:
            if os.path.exists(tmp):
                os.unlink(tmp)
        head = lines[0]
        body += cut(lines[1:], ref_id, n, opt["estimator"]) if n else lines[1:]
    cli.write_atomic(opt["out"], head + "".join(body))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
