"""Shared helpers for the test-suite: fixture decoding, byte packing, small point pools (exact big-int tier)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from constantine_b200.curves import CURVES  # noqa: E402
from oracle import pyref  # noqa: E402


def reference_c_api():
    """The reference's typedefs and prototypes of the names our header also declares, per reference header in include order
    (tests/golden/make_capi_golden.py)."""
    import json
    with open(os.path.join(ROOT, "tests", "golden", "reference_c_api.json")) as f:
        return json.load(f)["headers"]


def dec_point(p):
    if p is None:
        return None
    return (tuple(int(c, 16) for c in p[0]), tuple(int(c, 16) for c in p[1]))


def case_inputs(case):
    cv = CURVES[case["curve"]]
    ks = [int(s, 16) for s in case["scalars"]]
    pts = [dec_point(p) for p in case["points"]]
    return cv, ks, pts, dec_point(case["expected"])


def pack(cv, ks, pts, fr_mont=False):
    cb = b"".join(pyref.scalar_to_bytes(k, cv, fr_mont=fr_mont) for k in ks)
    pb = b"".join(pyref.aff_to_bytes(P, cv) for P in pts)
    return cb, pb


_pool_cache = {}


def point_pool(cv, size=48, seed=1):
    """`size` distinct subgroup points k_i*G with known k_i (exact tier)."""
    key = (cv.name, size, seed)
    if key not in _pool_cache:
        import random
        r = random.Random(seed)
        ks = [r.getrandbits(64) | 1 for _ in range(size)]
        _pool_cache[key] = (ks, [pyref.ec_mul_fast(k, cv.gen, cv) for k in ks])
    return _pool_cache[key]


def xyzz_bytes_to_affine(b, cv):
    """Raw XYZZ (x = X/ZZ, y = Y/ZZZ; infinity iff ZZ == 0) -> affine tuple."""
    p = cv.fp.modulus
    cb = cv.coord_bytes
    X, Y, ZZ, ZZZ = (pyref.coord_from_bytes(b[i * cb:(i + 1) * cb], cv) for i in range(4))
    if pyref.f_is_zero(ZZ):
        return None
    return (pyref.f_mul(X, pyref.f_inv(ZZ, p), p), pyref.f_mul(Y, pyref.f_inv(ZZZ, p), p))


def affine_to_xyzz_bytes(P, cv):
    if P is None:
        return bytes(4 * cv.coord_bytes)
    one = (1,) + (0,) * (cv.ext_degree - 1)
    return (pyref.coord_to_bytes(P[0], cv.fp) + pyref.coord_to_bytes(P[1], cv.fp) +
            pyref.coord_to_bytes(one, cv.fp) + pyref.coord_to_bytes(one, cv.fp))
