"""Checks that the plain sponge kernels compile to the same instructions in two builds.

    python tools/compare_sass.py OLD NEW [--kernels sponge_kernel,sponge_tiered_kernel,sponge_kernel2]

OLD and NEW are each an object or library with sm_100a code (e.g. capycrypt_b200/_lib/obj_*/sha3_api.o) or a source tree
of this project, whose csrc/sha3_api.cu is then compiled with the flags of capycrypt_b200/build.py into a temporary
directory.  Every instantiation of the named kernels is disassembled (cuobjdump -sass) and compared instruction by
instruction after constant-bank offsets (c[0x0][0x...], where kernel parameters live) are masked: a kernel whose parameter
struct grew at its end reads the same fields at the same offsets, and a second struct behind it moves.  Prints one line
per kernel and exits 1 when any of them differs in anything else, or is missing in one build.  No GPU needed.
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))


def _object(path: str, tmp: str, tag: str) -> str:
    if os.path.isfile(path):
        return path
    from capycrypt_b200.build import BASE_FLAGS, NVCC

    obj = os.path.join(tmp, f"{tag}_sha3_api.o")
    src = os.path.join(path, "capycrypt_b200", "csrc", "sha3_api.cu")
    subprocess.run([NVCC, *BASE_FLAGS, "-c", src, "-o", obj], check=True)
    return obj


def _functions(obj: str) -> dict[str, list[str]]:
    """mangled name -> normalised instructions"""
    out = subprocess.run(["cuobjdump", "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs: dict[str, list[str]] = {}
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if cur is not None and m:
            cur.append(re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][*]", m.group(1)))
    return funcs


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--kernels", default="sponge_kernel,sponge_tiered_kernel,sponge_kernel2")
    args = ap.parse_args()
    names = args.kernels.split(",")
    with tempfile.TemporaryDirectory() as tmp:
        old = _functions(_object(args.old, tmp, "old"))
        new = _functions(_object(args.new, tmp, "new"))
    pick = lambda fs: {k: v for k, v in fs.items() if any(re.match(rf"_ZN4capy{len(n)}{n}ILi\d+EEEv", k) for n in names)}
    old, new = pick(old), pick(new)
    bad = 0
    for k in sorted(set(old) | set(new)):
        if k not in old or k not in new:
            print(f"MISSING in {'old' if k not in old else 'new'}: {k}")
            bad += 1
            continue
        a, b = old[k], new[k]
        diff = sum(x != y for x, y in zip(a, b)) + abs(len(a) - len(b))
        print(f"{'same' if diff == 0 else 'DIFFERENT'}: {k} ({len(a)} / {len(b)} instructions, {diff} differ)")
        bad += diff != 0
    if not old:
        print("no matching kernels found")
        return 1
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
