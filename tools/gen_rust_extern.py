"""Prints the `extern "C"` block of rust/gpu.rs from include/capy_gpu.h (so the Rust shim binds every export with the
header's own parameter names and types), and exposes the two parsers tests/test_rust_shim.py compares.

usage: python tools/gen_rust_extern.py            # prints the block
"""
from __future__ import annotations

import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "capy_gpu.h")
RUST = os.path.join(ROOT, "rust", "gpu.rs")

C_INT_TYPES = {"int": "c_int", "uint32_t": "u32", "uint64_t": "u64", "size_t": "usize", "double": "f64"}
C_PTR_BASE = {"void": "c_void", "uint8_t": "u8", "uint32_t": "u32", "uint64_t": "u64", "int": "c_int", "char": "c_char",
              "capy_ctx": "CapyCtx", "capy_ed448_pub": "CapyEd448Pub", "capy_hasher": "CapyHasher", "double": "f64"}


def _strip_comments(src: str) -> str:
    return re.sub(r"/\*.*?\*/", "", src, flags=re.S)


def c_type_to_rust(t: str) -> str:
    """'const uint8_t*' -> '*const u8', 'capy_ctx**' -> '*mut *mut CapyCtx', 'uint64_t' -> 'u64'."""
    t = " ".join(t.replace("*", " * ").split())
    const = t.startswith("const ")
    if const:
        t = t[len("const "):]
    parts = t.split(" ")
    base, stars = parts[0], parts.count("*")
    if stars == 0:
        return C_INT_TYPES[base]
    r = C_PTR_BASE[base]
    for level in range(stars):
        r = ("*const " if (const and level == 0) else "*mut ") + r
    return r


def parse_header(path: str = HEADER) -> dict[str, tuple[str, list[tuple[str, str]]]]:
    """name -> (rust return type or '', [(param name, rust type)])"""
    src = _strip_comments(open(path).read())
    out = {}
    for m in re.finditer(r"(?m)^\s*((?:const\s+)?[A-Za-z_][A-Za-z0-9_]*\s*\**)\s*(capy_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", src):
        ret, name, args = m.group(1).strip(), m.group(2), " ".join(m.group(3).split())
        params = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                mm = re.match(r"(.*?)([A-Za-z_][A-Za-z0-9_]*)$", a)
                params.append((mm.group(2), c_type_to_rust(mm.group(1).strip())))
        out[name] = ("" if ret == "void" else c_type_to_rust(ret), params)
    return out


def parse_rust(path: str = RUST) -> dict[str, tuple[str, list[tuple[str, str]]]]:
    src = re.sub(r"//[^\n]*", "", open(path).read())
    m = re.search(r'extern\s+"C"\s*\{(.*?)\n\}', src, flags=re.S)
    out = {}
    for f in re.finditer(r"fn\s+(capy_[a-z0-9_]+)\s*\((.*?)\)\s*(?:->\s*([^;]+?))?\s*;", m.group(1), flags=re.S):
        params = []
        args = " ".join(f.group(2).split())
        if args:
            for a in args.split(","):
                a = a.strip()
                if not a:
                    continue
                nm, ty = a.split(":", 1)
                params.append((nm.strip(), " ".join(ty.split())))
        out[f.group(1)] = ((f.group(3) or "").strip(), params)
    return out


def render() -> str:
    lines = ['#[link(name = "capycrypt_gpu", kind = "static")]', 'extern "C" {']
    for name, (ret, params) in parse_header().items():
        sig = f"    fn {name}(" + ", ".join(f"{n}: {t}" for n, t in params) + ")" + (f" -> {ret}" if ret else "") + ";"
        # wrap at 118 columns like the rest of the file
        while len(sig) > 118:
            cut = sig.rfind(", ", 0, 118)
            lines.append(sig[: cut + 1])
            sig = " " * 8 + sig[cut + 2:]
        lines.append(sig)
    lines.append("}")
    return "\n".join(lines)


if __name__ == "__main__":
    print(render())
