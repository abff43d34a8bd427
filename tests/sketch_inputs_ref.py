"""skani sketch files (`DB/<name>.sketch`) as triangle and dist inputs, on top of the CPU references -- TEST
INFRASTRUCTURE ONLY.

`python tests/sketch_inputs_ref.py <skani argv>` is the CPU `skani` for these inputs (DESIGN.md section 3).  It rewrites
the argv into its FASTA form: every entry ending in .sketch -- a FASTA argument, a -q / -r value, or an entry of an -l /
--ql / --rl list (rewritten into a list file in a temporary directory) -- becomes the path its descriptor records, the
one its database's manifest names for the descriptor's genome ids; without -m, the databases' m is added as -m.  Then
tests/matrix_ref.py's main (which defers to tests/cli_forms_ref.py for everything but --full-matrix) runs the result.
Sketches from databases of different m, an -m that differs from theirs, or a sketch whose database mode (-i or not)
differs from its side's flag are refused as cli.UsageError, as the shim refuses them.
"""
import json
import os
import shutil
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def fasta_of(sketch):
    """(the FASTA path a descriptor stands for, checked against its database's manifest; its Descriptor)"""
    from skder_b200 import sketch_files

    d = sketch_files.Descriptor(sketch)
    with open(os.path.join(d.db, "manifest.json")) as f:
        man = json.load(f)
    assert all(man["paths"][g] == d.path for g in d.ids), sketch
    assert [man["names"][g] for g in d.ids] == d.names, sketch
    return d.path, d


def rewrite(argv, tmp):
    """the FASTA-form argv of `argv` (list files it names rewritten into tmp)"""
    from search_queries_ref import VALUED
    from skder_b200 import cli
    from skder_b200.sketch_files import is_sketch

    sub, opt = cli.parse_args(argv)
    ms, n = set(), [0]

    def fasta(entry, flag_key):
        if not is_sketch(entry):
            return entry
        path, d = fasta_of(entry)
        if d.per_sequence != opt[flag_key]:
            raise cli.UsageError("%s: database mode differs from the side's per-sequence flag" % entry)
        ms.add(d.m)
        return path

    ref_key, query_key = ("ref_per_seq", "query_per_seq") if sub == "dist" else ("per_seq", "per_seq")
    list_keys = {"-l": ref_key, "--rl": ref_key, "--ql": query_key}
    out, i = [sub], 1
    pos = 0
    while i < len(argv):
        a = argv[i]
        if a in VALUED:
            v = argv[i + 1]
            if a in list_keys:
                n[0] += 1
                v = os.path.join(tmp, "list%d.txt" % n[0])
                with open(v, "w") as f:
                    f.write("".join(fasta(e, list_keys[a]) + "\n" for e in cli.read_list(argv[i + 1])))
            out += [a, v]
            i += 2
        elif a in ("-q", "-r"):
            out.append(a)
            i += 1
            while i < len(argv) and not argv[i].startswith("-"):
                out.append(fasta(argv[i], query_key if a == "-q" else ref_key) if argv[i] else "")
                i += 1
        elif a and not a.startswith("-"):  # dist Q R...: the first positional is the query
            out.append(fasta(a, query_key if sub == "dist" and pos == 0 else ref_key))
            pos += 1
            i += 1
        else:
            out.append(a)
            i += 1
    if len(ms) > 1 or (ms and opt["marker_c_given"] and opt["marker_c"] not in ms):
        raise cli.UsageError("the sketches' m and the command's differ")
    if ms and not opt["marker_c_given"]:
        out += ["-m", str(ms.pop())]
    return out


def main(argv):
    import matrix_ref

    tmp = tempfile.mkdtemp(prefix="sketch_inputs_ref.")
    try:
        return matrix_ref.main(rewrite(argv, tmp))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
