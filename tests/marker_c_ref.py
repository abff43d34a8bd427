"""skani's -m marker compression on top of the CPU oracle -- TEST INFRASTRUCTURE ONLY.

The oracle takes the marker compression as a parameter (ora_params_t.marker_c: a canonical 21-mer is a marker iff its
hash is below UINT64_MAX / marker_c); this module only makes every oracle call that uses the default parameters use a
given one.  The oracle itself is unchanged.  `python tests/marker_c_ref.py <skani argv>` is the CPU `skani` of
tests/oracle_skani.py (with tests/ani_estimators_ref.py, ani_ci_ref.py and ani_detail_ref.py for --median / --robust,
--ci and --detailed) run at the argv's -m.  `sketch -m M` records M in the database's manifest; `search` reads the
database's M from its sketches.skb when there is one (a database the B200 shim wrote), from the manifest otherwise.
"""
import contextlib
import json
import os
import struct
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import oracle as O  # noqa: E402

DEFAULT = 1000
_default_params = O.default_params


def params(m):
    """the oracle's default parameters at marker compression m"""
    p = _default_params()
    p.marker_c = m
    return p


@contextlib.contextmanager
def marker_c(m):
    """every oracle call inside that takes the default parameters sketches markers at compression m"""
    O.default_params = lambda: params(m)
    try:
        yield
    finally:
        O.default_params = _default_params


def db_marker_c(db):
    """the marker compression of a database directory: sketches.skb's header (SKB200v1: 1000; SKB200v2: the u64 after
    the magic), else the manifest's "marker_c" (a database this module sketched), else 1000"""
    path = os.path.join(db, "sketches.skb")
    if os.path.exists(path):
        with open(path, "rb") as f:
            head = f.read(16)
        if head[:8] == b"SKB200v2":
            return struct.unpack("<Q", head[8:16])[0]
        assert head[:8] == b"SKB200v1", head[:8]
        return DEFAULT
    with open(os.path.join(db, "manifest.json")) as f:
        return json.load(f).get("marker_c", DEFAULT)


def without_m(argv):
    out, i = [], 0
    while i < len(argv):
        if argv[i] == "-m":
            i += 2
            continue
        out.append(argv[i])
        i += 1
    return out


def main(argv):
    import ani_detail_ref
    import ani_estimators_ref
    from skder_b200 import cli

    sub, opt = cli.parse_args(argv)
    m = db_marker_c(opt["db"]) if sub == "search" else opt["marker_c"]
    rest = without_m(argv)
    with marker_c(m):
        # ani_detail_ref falls through to ani_ci_ref, and that to oracle_skani, when its flag is absent
        rc = (ani_estimators_ref if opt["estimator"] != "mean" else ani_detail_ref).main(rest)
    if rc == 0 and sub == "sketch" and m != DEFAULT:
        man = os.path.join(opt["out"], "manifest.json")
        with open(man) as f:
            d = json.load(f)
        cli.write_atomic(man, json.dumps(dict(d, marker_c=m)))
    return rc


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
