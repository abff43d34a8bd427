"""skani's --median and --robust ANI estimators restated on top of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

The oracle (oracle/skani_oracle.c ora_pair) computes the pooled mean and hands out the pair's accepted chains; this
module turns those chains into the median or robust ANI exactly as DESIGN.md section 3 defines them, with the same
integer key and the same double arithmetic as the device (est_key_kernel / est_pick_kernel), and leaves every other
field of the oracle's result as it is.  `python tests/ani_estimators_ref.py <skani argv>` is tests/oracle_skani.py
(the CPU `skani`) with the estimator the argv names.
"""
import contextlib
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402

MODES = ("mean", "median", "robust")
_oracle_pair = O.pair


def chosen_counts(chains, mode):
    """(anchors, seeds) whose ratio is `mode`'s estimate: chains ranked by the key (a << 47) // s with a = n_anchors - 2,
    s = n_seeds - 2, ties by (chunk, score desc, q0, r0), weighted by s."""
    ch = sorted(((((c.n_anchors - 2) << 47) // (c.n_seeds - 2), c.chunk, -c.score, c.q0, c.r0), c.n_anchors - 2,
                 c.n_seeds - 2) for c in chains)
    W = sum(s for _, _, s in ch)
    if mode == "mean":
        return sum(a for _, a, _ in ch), W
    C_, sa, ss = 0, 0, 0
    for _, a, s in ch:
        C_ += s
        if mode == "median" and 2 * C_ >= W:
            return a, s
        if mode == "robust" and 10 * C_ > W and 10 * (C_ - s) < 9 * W:
            sa, ss = sa + a, ss + s
    return sa, ss


def debias(raw):
    f = O.lib().ora_debias
    f.restype, f.argtypes = C.c_double, [C.c_double]
    return f(raw)


def pair(a, b, params=None, mode="mean"):
    """oracle.pair with `mode`'s ANI: ani_raw = (chosen anchors / chosen seeds)^(1/15), ani = the debias substitute of it;
    AF, chain / anchor / seed counts and spans are the oracle's (the totals over all accepted chains)."""
    r = _oracle_pair(a, b, params)
    if mode == "mean" or r.ani < 0:
        return r
    _, chains = _oracle_pair(a, b, params, want_chains=True, max_chains=max(1, r.n_chains))
    n, d = chosen_counts(chains, mode)
    r.ani_raw = min(1.0, n / d) ** (1.0 / 15)
    r.ani = min(1.0, debias(r.ani_raw))
    return r


@contextlib.contextmanager
def estimator(mode):
    """every oracle.pair call inside (oracle/skani_cpu.py, tests/oracle_skani.py) gives `mode`'s ANI"""
    O.pair = lambda a, b, params=None, want_chains=False, max_chains=8192: (
        _oracle_pair(a, b, params, want_chains, max_chains) if want_chains else pair(a, b, params, mode))
    try:
        yield
    finally:
        O.pair = _oracle_pair


def main(argv):
    import oracle_skani
    from skder_b200 import cli

    with estimator(cli.parse_args(argv)[1]["estimator"]):
        return oracle_skani.main(argv)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
