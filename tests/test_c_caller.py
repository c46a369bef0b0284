"""A plain C program (tests/c_api/msm_smoke.c) that includes include/ctt_b200_msm.h and calls the reference-named symbol:
the drop-in boundary exercised from C, not through Python."""
import os
import subprocess

import pytest

from helpers import CURVES, ROOT, pyref, reference_c_api

SRC = os.path.join(ROOT, "tests", "c_api", "msm_smoke.c")
LIBDIR = os.path.join(ROOT, "constantine_b200", "lib")


def _build(tmp_path, src=None, name="msm_smoke"):
    exe = str(tmp_path / name)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), src or SRC,
                           "-L", LIBDIR, "-lctt_b200_msm", f"-Wl,-rpath,{LIBDIR}", "-o", exe])
    return exe


def test_c_program_compiles_links_and_uses_the_threadpool_handle(tmp_path):
    exe = _build(tmp_path)
    out = subprocess.run([exe, "--link-only"], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0 and "linked ok" in out.stdout


def test_header_coexists_with_the_reference_headers(tmp_path):
    """Both header sets in one translation unit (type definitions are guarded, prototypes must agree). The reference's
    bls12_381 / bn254_snarks / pallas / vesta _parallel.h headers and what they include are replayed, under their own include
    guards and in their include order, from their declarations of the names our header declares too
    (tests/golden/reference_c_api.json)."""
    lines = ["#include <stddef.h>", "#include <stdint.h>"]
    for h in reference_c_api():
        lines += [f"#ifndef {h['guard']}", f"#define {h['guard']}", *h["typedefs"], *h["prototypes"], "#endif"]
    src = tmp_path / "both.c"
    src.write_text("\n".join(lines) + '\n#include "ctt_b200_msm.h"\nint main(void) { return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])


@pytest.mark.gpu
def test_c_program_result_matches_the_eip2537_vector(tmp_path, kat):
    exe = _build(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    limbs = [int(x, 16) for x in out.stdout.split()]
    assert len(limbs) == 18
    raw = b"".join(v.to_bytes(8, "little") for v in limbs)
    cv = CURVES["bls12_381_g1"]
    case = next(c for c in kat["eip2537"] if c["name"] == "bls_g1multiexp_(g1+g1=2*g1)")
    want = (tuple(int(c, 16) for c in case["expected"][0]), tuple(int(c, 16) for c in case["expected"][1]))
    assert pyref.jac_bytes_to_affine(raw, cv) == want


@pytest.mark.gpu
def test_c_program_multi_gpu_behind_the_unchanged_symbol(tmp_path):
    """tests/c_api/msm_multi_gpu.c: malloc'd inputs, the reference symbol once on one device and once with the device list set
    (every visible GPU; one GPU listed twice on a one-GPU box) -- both equal the closed form [N (N + 1) / 2] G."""
    exe = _build(tmp_path, os.path.join(ROOT, "tests", "c_api", "msm_multi_gpu.c"), "msm_multi_gpu")
    n = 100000
    out = subprocess.run([exe, str(n)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    toks = out.stdout.split()
    assert toks[-2] == "devices" and int(toks[-1]) >= 2
    limbs = [int(x, 16) for x in toks[:36]]
    cv = CURVES["bls12_381_g1"]
    want = pyref.ec_mul_fast(n * (n + 1) // 2 % cv.fr.modulus, cv.gen, cv)
    for k in range(2):
        raw = b"".join(v.to_bytes(8, "little") for v in limbs[18 * k:18 * k + 18])
        assert pyref.jac_bytes_to_affine(raw, cv) == want, k
