"""skani's --ci interval restated on top of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

The oracle (oracle/skani_oracle.c ora_pair) hands out a pair's accepted chains; this module turns them into the
percentile-bootstrap interval of the mean ANI exactly as DESIGN.md section 3 defines it: Python integers for the draws,
the replicate sums and the ranking, then the device's double arithmetic for the two bounds.  The oracle itself is
unchanged.  `python tests/ani_ci_ref.py <skani argv>` is tests/oracle_skani.py (the CPU `skani`); with --ci every row
gains the two interval columns.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402

REPS, LO, HI = 100, 5, 94
M64 = (1 << 64) - 1


def mix(z):
    """splitmix64 finalizer, mod 2^64"""
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def canonical(chains):
    """[(a, s)] of the accepted chains in (chunk, score desc, q0, r0) order; a = n_anchors - 2, s = n_seeds - 2"""
    return [(c.n_anchors - 2, c.n_seeds - 2) for c in sorted(chains, key=lambda c: (c.chunk, -c.score, c.q0, c.r0))]


def replicates(chains):
    """[(A_b, S_b)] for b = 0 .. REPS-1"""
    ch = canonical(chains)
    n, A, S = len(ch), sum(a for a, _ in ch), sum(s for _, s in ch)
    seed = mix(mix(mix(n) ^ A) ^ S)
    out = []
    for b in range(REPS):
        sa = ss = 0
        for i in range(n):
            a, s = ch[(mix(seed ^ (b << 40) ^ i) * n) >> 64]
            sa += a
            ss += s
        out.append((sa, ss))
    return out


def picks(reps):
    """(A, S) of the replicates at ranks LO and HI: ranked by A/S (cross products), ties by b; rank = how many sort
    before"""
    got = {}
    for x, (ax, sx) in enumerate(reps):
        rank = sum(1 for y, (ay, sy) in enumerate(reps) if ay * sx < ax * sy or (ay * sx == ax * sy and y < x))
        if rank in (LO, HI):
            got[rank] = (ax, sx)
    return got[LO], got[HI]


def debias(raw):
    import ctypes as C

    f = O.lib().ora_debias
    f.restype, f.argtypes = C.c_double, [C.c_double]
    return f(raw)


def bound(a, s):
    """the ANI of a ratio a / s (fraction), as the mean's: min(1, a/s)^(1/15), then the debias substitute"""
    return min(1.0, debias(min(1.0, a / s) ** (1.0 / 15)))


def interval(x, y, params=None):
    """(lo, hi) ANI fractions of the pair (x, y), or None when it has no estimate"""
    r = O.pair(x, y, params)
    if r.ani < 0:
        return None
    _, chains = O.pair(x, y, params, want_chains=True, max_chains=max(1, r.n_chains))
    lo, hi = picks(replicates(chains))
    return bound(*lo), bound(*hi)


def main(argv):
    import oracle_skani
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)
    if not opt["ci"]:
        return oracle_skani.main(argv)
    rc = oracle_skani.main([a for a in argv if a != "--ci"])
    if rc or sub == "sketch":
        return rc
    with open(opt["out"]) as f:
        lines = f.read().splitlines()
    sk = {}
    out = [cli.header(True)]
    for ln in lines[1:]:
        t = ln.split("\t")
        for p in t[:2]:
            if p not in sk:
                sk[p] = O.Sketch.from_file(p)
        out.append(ln + "\t%.2f\t%.2f\n" % tuple(100.0 * v for v in interval(sk[t[0]], sk[t[1]])))
    cli.write_atomic(opt["out"], "".join(out))
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
