"""skani's --detailed columns restated on top of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

The oracle (oracle/skani_oracle.c ora_pair) hands out a pair's accepted chains and its AF numerators; this module turns
them into the per-edge values of the 13 --detailed columns as DESIGN.md section 3 defines them: the --ci interval
(tests/ani_ci_ref.py), the seed-weighted standard deviation of the per-chain ANI (two passes, Python floats), the
covered bases of both genomes, and Nx over each genome's kept contigs.  The oracle itself is unchanged.
`python tests/ani_detail_ref.py <skani argv>` is tests/ani_ci_ref.py (the CPU `skani`, with --ci); with --detailed
every row gains the 13 columns instead.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import ani_ci_ref as CI  # noqa: E402
from oracle import oracle as O  # noqa: E402


def chain_sd(chains):
    """the seed-weighted standard deviation (fraction) of the chains' own ANI: d_c = the ANI of (a_c, s_c) alone,
    mu = sum s_c d_c / W, sd = sqrt(sum s_c (d_c - mu)^2 / W); 0 for one chain"""
    ch = CI.canonical(chains)
    if len(ch) == 1:
        return 0.0
    d = [CI.bound(a, s) for a, s in ch]
    W = float(sum(s for _, s in ch))
    mu = sum(s * x for (_, s), x in zip(ch, d)) / W
    return (sum(s * (x - mu) ** 2 for (_, s), x in zip(ch, d)) / W) ** 0.5


def nx(sketch):
    """(N90, N50, N10) over the kept contigs: lengths descending, the first l_k with 100 (l_1 + ... + l_k) >= x T"""
    lens = sorted((int(v) for v in sketch.contig_lens()), reverse=True)
    total, out = sum(lens), []
    for x in (90, 50, 10):
        cum, v = 0, 0
        for ln in lens:
            cum += ln
            if 100 * cum >= x * total:
                v = ln
                break
        out.append(v)
    return tuple(out)


def detail(x, y, params=None):
    """{lo, hi, sd (fractions), covered_a, covered_b, n_chains} of the pair (x = edge a, y = edge b), or None when it
    has no estimate"""
    r = O.pair(x, y, params)
    if r.ani < 0:
        return None
    _, chains = O.pair(x, y, params, want_chains=True, max_chains=max(1, r.n_chains))
    lo, hi = CI.picks(CI.replicates(chains))
    return {"lo": CI.bound(*lo), "hi": CI.bound(*hi), "sd": chain_sd(chains),
            "covered_a": r.span_r if r.swapped else r.span_q, "covered_b": r.span_q if r.swapped else r.span_r,
            "n_chains": r.n_chains}


def columns(x, y, params=None):
    """the 13 --detailed values of the row (Ref = x, Query = y), in cli.DETAILED_COLUMNS order"""
    d = detail(x, y, params)
    return ((x.n_contigs, y.n_contigs, 100.0 * d["lo"], 100.0 * d["hi"], 100.0 * d["sd"]) + nx(x) + nx(y) +
            (d["covered_b"] // d["n_chains"], d["covered_b"]))


def main(argv):
    import oracle_skani
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)
    if not opt["detailed"]:
        return CI.main(argv)
    rc = oracle_skani.main([a for a in argv if a not in ("--ci", "--detailed")])
    if rc or sub == "sketch":
        return rc
    with open(opt["out"]) as f:
        lines = f.read().splitlines()
    sk = {}
    out = [cli.header(opt["ci"], True)]
    for ln in lines[1:]:
        t = ln.split("\t")
        for p in t[:2]:
            if p not in sk:
                sk[p] = O.Sketch.from_file(p)
        out.append(ln + cli.DETAILED_FMT % columns(sk[t[0]], sk[t[1]]))
    cli.write_atomic(opt["out"], "".join(out))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
