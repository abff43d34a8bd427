"""Downstream replay: edge list -> representatives with the reference's selection rules.

greedy : skDERsum (reference src/skDER/skDERsum.cpp), restated in greedy_information below and held to the reference's
         own output (tests/golden/skder_results/Genome_Information_for_Greedy_Clustering.txt byte for byte, and the
         representatives of all 31 golden runs, tests/test_downstream_and_multi.py)
         -> `sort -k 2 -gr` -> the loop of reference src/skDER/skder.py:150-165, restated below.
dynamic: skDERcore (reference src/skDER/skDERcore.cpp, compiled into oracle/_ref by oracle/build_ref.py where the
         reference is available), as reference src/skDER/skder.py:78-80 runs it.
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def helpers():
    from oracle import build_ref

    return build_ref.build()


def greedy_information(edge_tsv, n50_tsv, ani, af):
    """What `skDERsum <edge TSV> <N50 TSV> <ANI> <AF>` prints: one row per genome of the N50 file, in its order -- the
    genome, N50 x the number of genomes it covers (C++ `ostream << double`, i.e. %g), and those genomes joined by "; ".
    A row (Ref, Query, ANI, AF_ref, AF_query) with ANI >= ani makes Ref cover Query when AF_query >= af and Query cover
    Ref when AF_ref >= af; members are listed in the order of the rows that made them.  A genome covering nothing
    prints "0.0" and no members."""
    members = {}
    with open(edge_tsv) as f:
        next(f)
        for line in f:
            t = line.rstrip("\n").split("\t")
            if float(t[2]) >= ani:
                if float(t[4]) >= af:
                    members.setdefault(t[0], []).append(t[1])
                if float(t[3]) >= af:
                    members.setdefault(t[1], []).append(t[0])
    out = []
    with open(n50_tsv) as f:
        for line in f:
            if not line.strip():
                continue
            path, n50 = line.rstrip("\n").split("\t")[:2]
            m = members.get(path)
            out.append("%s\t%g\t%s\n" % (path, float(int(n50)) * len(m), "; ".join(m)) if m else path + "\t0.0\t\n")
    return "".join(out)


def sorted_greedy_information(gi_path, workdir):
    """The reference's own sort of the summary (skder.py:146): `sort -k 2 -gr`, C locale."""
    srt = os.path.join(workdir, "gi.sorted.txt")
    with open(srt, "w") as f:
        subprocess.check_call(["sort", "-k", "2", "--parallel=2", "-gr", gi_path], stdout=f, env=dict(os.environ, LC_ALL="C"))
    return srt


def greedy_reps(edge_tsv, n50_tsv, ani, af, workdir):
    gi = os.path.join(workdir, "gi.txt")
    with open(gi, "w") as f:
        f.write(greedy_information(edge_tsv, n50_tsv, ani, af))
    srt = sorted_greedy_information(gi, workdir)
    reps, accounted = [], set()
    with open(srt) as f:  # reference skder.py:150-165
        for line in f:
            ls = line.rstrip("\n").split("\t")
            if ls[0] in accounted:
                continue
            reps.append(ls[0])
            accounted.add(ls[0])
            if len(ls) > 2 and ls[2].strip():
                for m in ls[2].split("; "):
                    accounted.add(m.strip())
    return reps


def dynamic_reps(edge_tsv, n50_tsv, ani, af, max_af_diff):
    h = helpers()
    out = subprocess.check_output([h["skDERcore"], edge_tsv, n50_tsv, str(ani), str(af), str(max_af_diff)], text=True)
    return [ln for ln in out.splitlines() if ln.strip()]
