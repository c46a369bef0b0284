"""CPU: the C-ABI shared library loads and exports every symbol include/ctt_b200_msm.h declares (no compute calls)."""
import ctypes
import os
import re

from helpers import ROOT, reference_c_api


def _declared_functions():
    hdr = open(os.path.join(ROOT, "include", "ctt_b200_msm.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(ctt_[a-z0-9_]+)\s*\(", hdr))
    return names


def test_header_declares_the_reference_family():
    names = _declared_functions()
    for curve in ("bls12_381_g1", "bn254_snarks_g1", "pallas_ec", "vesta_ec"):
        for out in ("jac", "prj"):
            for kind in ("big", "fr"):
                # reference include/constantine/curves/*_parallel.h:21-24 and the serial twins
                assert f"ctt_{curve}_{out}_multi_scalar_mul_{kind}_coefs_vartime_parallel" in names
                assert f"ctt_{curve}_{out}_multi_scalar_mul_{kind}_coefs_vartime" in names
    for curve in ("bls12_381_g2", "bn254_snarks_g2"):
        for out in ("jac", "prj"):
            for kind in ("big", "fr"):
                assert f"ctt_{curve}_{out}_multi_scalar_mul_{kind}_coefs_vartime" in names


def test_library_exports_every_declared_symbol():
    from constantine_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_functions()
    listed = set(open(os.path.join(ROOT, "include", "exported_symbols.txt")).read().split())
    assert declared == listed
    assert len(declared) >= 64
    for name in sorted(declared):
        assert hasattr(lib, name), name


def test_reference_headers_prototypes_match_when_available():
    """Our prototypes of the 16 _parallel symbols are textually the reference's generated ones
    (include/constantine/curves/*_parallel.h, stored in tests/golden/reference_c_api.json)."""
    ours = open(os.path.join(ROOT, "include", "ctt_b200_msm.h")).read()
    norm = lambda s: re.sub(r"\s+", " ", s).strip()
    ours_n = norm(ours)
    lines = [p for h in reference_c_api() if h["file"].endswith("_parallel.h") for p in h["prototypes"] if "multi_scalar_mul" in p]
    assert len(lines) == 16
    for line in lines:
        assert norm(line) in ours_n, line


def test_threadpool_handle_and_plan_need_no_gpu():
    from constantine_b200 import msm as M
    tp = M.Threadpool.new(4)
    assert tp._h
    tp.shutdown()
    c, w = M.plan("bls12_381_g1", 1 << 20)
    assert 10 <= c <= 20 and w == 255 // c + 1
    c, w = M.plan("bn254_snarks_g1", 256, force_c=7)
    assert (c, w) == (7, 37)  # reference: BN254 N=256 -> c=7, 37 windows (SURVEY.md Appendix C)
