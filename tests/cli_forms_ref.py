"""skani's positional, -q / -r and standard-output command forms on top of the CPU references -- TEST INFRASTRUCTURE
ONLY.

`python tests/cli_forms_ref.py <skani argv>` is the CPU `skani` for these forms (DESIGN.md section 3).  It rewrites the
argv into the list-file form the other references read: the FASTA arguments and -q / -r values go into list files in a
temporary directory, in the order the rules give them --
  triangle: `-l` = the FASTA arguments, then the -l entries (the triangle reference deduplicates and sorts);
  sketch:   `-l` = the FASTA arguments, then the -l entries;
  dist:     `--ql` = the -q values, then the --ql entries, `--rl` likewise; or for `dist Q R1 [R2 ...]`, `--ql` = Q and
            `--rl` = R1 R2 ...;
  search:   unchanged (the references take its positional queries)
-- and runs tests/per_sequence_ref.py's main, the outermost reference, on it.  Without -o the output goes to a file in
that directory and is copied to stdout when the run succeeds.  The references themselves are unchanged.
"""
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def rewrite(argv, tmp):
    """(the list-file argv of `argv`, with -o set to a file in tmp when argv has none; whether argv had -o).
    Raises cli.UsageError for an argv the shim refuses."""
    from search_queries_ref import VALUED
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)

    def listfile(name, entries):
        p = os.path.join(tmp, name)
        with open(p, "w") as f:
            f.write("".join(e + "\n" for e in entries))
        return p

    def listed(key):
        return cli.read_list(opt[key]) if key in opt else []

    pos = opt["positional"]
    if sub in ("triangle", "sketch"):
        lists = {"-l": listfile("l.txt", pos + listed("list"))}
    elif sub == "dist" and pos:
        lists = {"--ql": listfile("ql.txt", pos[:1]), "--rl": listfile("rl.txt", pos[1:])}
    elif sub == "dist":
        lists = {"--ql": listfile("ql.txt", opt.get("q", []) + listed("ql")),
                 "--rl": listfile("rl.txt", opt.get("r", []) + listed("rl"))}
    else:
        lists = {}
    out, i = [sub], 1
    while i < len(argv):
        a = argv[i]
        if a in VALUED:
            if a not in lists:
                out += argv[i:i + 2]
            i += 2
        elif a in ("-q", "-r"):  # its values run up to the next argument starting with '-'
            i += 1
            while i < len(argv) and not argv[i].startswith("-"):
                i += 1
        elif lists and a and not a.startswith("-"):  # a FASTA argument, now in a list file
            i += 1
        else:
            out.append(a)
            i += 1
    for a, p in lists.items():
        out += [a, p]
    has_out = "out" in opt
    if not has_out:
        out += ["-o", os.path.join(tmp, "out.tsv")]
    return out, has_out


def main(argv):
    import per_sequence_ref

    tmp = tempfile.mkdtemp(prefix="cli_forms_ref.")
    try:
        list_argv, has_out = rewrite(argv, tmp)
        rc = per_sequence_ref.main(list_argv)
        if rc == 0 and not has_out:
            with open(os.path.join(tmp, "out.tsv"), "rb") as f:
                data = f.read()
            sys.stdout.flush()
            sys.stdout.buffer.write(data)
            sys.stdout.flush()
        return rc
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
