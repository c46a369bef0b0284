#!/usr/bin/env python3
"""Extract the reference's C declarations of the names include/ctt_b200_msm.h also declares.

    python tests/golden/make_capi_golden.py <constantine checkout>/include

Reads the reference's four `<curve>_parallel.h` headers and everything they include, in the order a C compiler first sees them.
For each header it keeps the include guard and the typedefs and function prototypes of names our header declares too
(whitespace normalised, CTT_WORDS_REQUIRED(bits) evaluated for 64-bit words). Output: tests/golden/reference_c_api.json, which
tests/test_c_caller.py and tests/test_capi_symbols.py replay to check that both header sets compile in one translation unit and
that our prototypes are the reference's.
"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TOP = ["constantine/curves/bls12_381_parallel.h", "constantine/curves/bn254_snarks_parallel.h",
       "constantine/curves/pallas_parallel.h", "constantine/curves/vesta_parallel.h"]
STD_TYPES = {"size_t", "ptrdiff_t", "uint8_t", "uint32_t", "uint64_t"}


def strip_comments(text):
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def statements(text):
    """Top-level C statements ending in ';' (preprocessor lines and extern "C" braces dropped), whitespace normalised."""
    body = []
    for line in text.splitlines():
        s = line.strip()
        if s.startswith("#") or s in ('extern "C" {', "}"):
            continue
        body.append(s)
    out, cur, depth = [], "", 0
    for ch in " ".join(body):
        cur += ch
        depth += (ch == "{") - (ch == "}")
        if ch == ";" and depth == 0:
            out.append(re.sub(r"\s+", " ", cur).strip())
            cur = ""
    return out


def main():
    inc = sys.argv[1]
    ours = strip_comments(open(os.path.join(ROOT, "include", "ctt_b200_msm.h")).read())
    our_names = set(re.findall(r"\b[A-Za-z_]\w*\b", ours))
    order, seen = [], set()

    def visit(rel):
        if rel in seen:
            return
        seen.add(rel)
        text = strip_comments(open(os.path.join(inc, rel)).read())
        for dep in re.findall(r'#include\s+"([^"]+)"', text):
            visit(dep)
        order.append((rel, text))

    for rel in TOP:
        visit(rel)
    headers = []
    for rel, text in order:
        guard = re.search(r"#ifndef\s+(\w+)", text).group(1)
        typedefs, prototypes = [], []
        for st in statements(text):
            st = re.sub(r"CTT_WORDS_REQUIRED\((\d+)\)", lambda m: str((int(m.group(1)) + 63) // 64), st)
            if st.startswith("typedef "):
                name = re.search(r"(\w+)\s*;$", st).group(1)
                if name in our_names and name not in STD_TYPES:
                    typedefs.append(st)
            else:
                m = re.search(r"\b(ctt_\w+)\s*\(", st)
                if m and m.group(1) in our_names:
                    prototypes.append(st)
        headers.append({"file": rel, "guard": guard, "typedefs": typedefs, "prototypes": prototypes})
    out = {"source": "mratsim/constantine e6bee85e8c7a89af279460e4ca03283d817d1ce9, include/ (64-bit words)", "headers": headers}
    path = os.path.join(HERE, "reference_c_api.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", path, sum(len(h["typedefs"]) for h in headers), "typedefs,", sum(len(h["prototypes"]) for h in headers), "prototypes")


if __name__ == "__main__":
    main()
