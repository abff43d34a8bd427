"""skani's `triangle --full-matrix [--distance]` on top of the CPU references -- TEST INFRASTRUCTURE ONLY.

`python tests/matrix_ref.py <skani argv>` is the CPU `skani` for these flags (DESIGN.md section 3).  It rewrites the argv
to the -E form (--full-matrix and --distance dropped, -E added, -o pointed at a temporary TSV), runs
tests/cli_forms_ref.py's main on it, and renders both matrices from that TSV's text: every off-diagonal cell is a column
of an -E row, so the TSV and the genome labels are all it needs.  Outputs are placed as the shim places them: the ANI
matrix in -o or on stdout, the AF matrix in OUT.af or ./skani_matrix.af.  Any other argv goes to cli_forms_ref as is.
"""
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def genomes(opt):
    """(labels, keys) of the triangle's genomes in id order: a key is what an -E row names a genome by -- its path, or
    with -i its (path, record header) -- and a label is what the matrix rows show: the path, or with -i the header"""
    import per_sequence_ref
    from skder_b200 import cli

    paths = cli.inputs("triangle", opt)
    if not opt["per_seq"]:
        return paths, paths
    keys = [(p, name) for p in paths for name, _ in per_sequence_ref.records(p)]
    return [name for _, name in keys], keys


def cents(text):
    """the hundredths of a printed `%.2f` value"""
    return int(text.replace(".", ""))


def matrices(tsv, labels, keys, per_seq, distance=False):
    """(ANI or --distance matrix text, AF matrix text) from an -E TSV's text"""
    idx = {k: i for i, k in enumerate(keys)}
    assert len(idx) == len(keys), "genome keys must be unique"
    n = len(keys)
    ani = [["0.00"] * n for _ in range(n)]
    af = [["0.00"] * n for _ in range(n)]
    for i in range(n):
        ani[i][i] = af[i][i] = "100.00"
    for line in tsv.splitlines()[1:]:
        t = line.split("\t")
        a, b = (idx[(t[col], t[name]) if per_seq else t[col]] for col, name in ((0, 5), (1, 6)))
        ani[a][b] = ani[b][a] = t[2]
        af[a][b], af[b][a] = t[3], t[4]
    if distance:
        ani = [["%d.%02d" % divmod(10000 - cents(x), 100) for x in row] for row in ani]

    def text(m):
        return "%d\n" % n + "".join(lb + "".join("\t" + x for x in row) + "\n" for lb, row in zip(labels, m))

    return text(ani), text(af)


def main(argv):
    import cli_forms_ref
    import per_sequence_ref
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)
    if not opt["full_matrix"]:
        return cli_forms_ref.main(argv)
    tmp = tempfile.mkdtemp(prefix="matrix_ref.")
    try:
        tsv = os.path.join(tmp, "edges.tsv")
        rc = cli_forms_ref.main(per_sequence_ref.replace(argv, {"-o": tsv}, ("--full-matrix", "--distance")) + ["-E"])
        if rc:
            return rc
        with open(tsv) as f:
            labels, keys = genomes(opt)
            ani, af = matrices(f.read(), labels, keys, opt["per_seq"], opt["distance"])
        cli.write_atomic(opt["out"] + ".af" if "out" in opt else "skani_matrix.af", af)
        if "out" in opt:
            cli.write_atomic(opt["out"], ani)
        else:
            sys.stdout.flush()
            sys.stdout.buffer.write(ani.encode())
            sys.stdout.flush()
        return 0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
