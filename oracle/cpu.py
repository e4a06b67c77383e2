"""ctypes loader for the C oracle (oracle/ref_cpu.c).  TEST INFRASTRUCTURE ONLY.

Importable from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs; never from capycrypt_b200/.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_u8p = C.POINTER(C.c_uint8)
_u64p = C.POINTER(C.c_uint64)
_NATIVE_DIR = None


def build(native: bool = False, force: bool = False) -> str:
    """Compile ref_cpu.c.  native=True adds -march=native (bench CPU-baseline leg, built on
    the machine that times it); the default x86-64-v3 build runs on any x86-64-v3 host.
    The native build happens at benchmark time, when the tree may be read-only, so it goes to
    a temporary directory that lives as long as the process."""
    global _NATIVE_DIR
    if native:
        if _NATIVE_DIR is None:
            _NATIVE_DIR = tempfile.TemporaryDirectory(prefix="capy_oracle_")
        out = os.path.join(_NATIVE_DIR.name, "libcapy_oracle_native.so")
    else:
        out = os.path.join(_HERE, "_build", "libcapy_oracle.so")
    src = os.path.join(_HERE, "ref_cpu.c")
    if force or not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(src):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        march = "native" if native else "x86-64-v3"
        cmd = ["gcc", "-O3", f"-march={march}", "-fopenmp", "-fPIC", "-std=c11", "-shared", "-o", out, src]
        subprocess.run(cmd, check=True, capture_output=True)
    return out


def _p8(a):
    return a.ctypes.data_as(_u8p) if a is not None else None


def _p64(a):
    return a.ctypes.data_as(_u64p)


def _u8(b) -> np.ndarray:
    if isinstance(b, np.ndarray):
        return np.ascontiguousarray(b, dtype=np.uint8).reshape(-1)
    return np.frombuffer(bytes(b), dtype=np.uint8).copy() if len(b) else np.zeros(0, np.uint8)


def pack(items) -> tuple[np.ndarray, np.ndarray]:
    """list of bytes -> (packed u8 array (>=1 byte), u64 offsets[n+1])."""
    off = np.zeros(len(items) + 1, dtype=np.uint64)
    if len(items):
        off[1:] = np.cumsum([len(x) for x in items], dtype=np.uint64)
    data = np.frombuffer(b"".join(bytes(x) for x in items) or b"\0", dtype=np.uint8).copy()
    return data, off


class Oracle:
    def __init__(self, native: bool = False):
        self.lib = C.CDLL(build(native=native))
        self.max_threads = self.lib.capy_ref_max_threads()

    # ---- SHA3 side ----
    def keccakf(self, lanes):
        a = np.array(lanes, dtype=np.uint64)
        self.lib.capy_ref_keccakf(_p64(a))
        return a

    def sha3_batch(self, data, off, d, threads=1, lean=0):
        data, off = _u8(data), np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        out = np.zeros((n, d // 8), dtype=np.uint8)
        rc = self.lib.capy_ref_sha3_batch(_p8(data), _p64(off), C.c_uint64(n), d, _p8(out), threads, lean)
        if rc:
            raise ValueError(f"oracle rc={rc}")
        return out

    def sha3(self, msg: bytes, d: int) -> bytes:
        data, off = pack([msg])
        return self.sha3_batch(data, off, d)[0].tobytes()

    def cshake_batch(self, data, off, l_bits, n_str, s_str, d, threads=1, lean=0):
        data, off = _u8(data), np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        out = np.zeros((n, l_bits // 8), dtype=np.uint8)
        nn, ss = _u8(n_str), _u8(s_str)
        rc = self.lib.capy_ref_cshake_batch(_p8(data), _p64(off), C.c_uint64(n), C.c_size_t(l_bits), _p8(nn),
                                            C.c_size_t(len(nn)), _p8(ss), C.c_size_t(len(ss)), d, _p8(out), threads, lean)
        if rc:
            raise ValueError(f"oracle rc={rc}")
        return out

    def kmac_xof_batch(self, keys, koff, data, off, l_bits, s_str, d, threads=1, lean=0):
        keys, koff = _u8(keys), np.ascontiguousarray(koff, dtype=np.uint64)
        data, off = _u8(data), np.ascontiguousarray(off, dtype=np.uint64)
        n = len(off) - 1
        out = np.zeros((n, l_bits // 8), dtype=np.uint8)
        ss = _u8(s_str)
        rc = self.lib.capy_ref_kmac_xof_batch(_p8(keys), _p64(koff), _p8(data), _p64(off), C.c_uint64(n),
                                              C.c_size_t(l_bits), _p8(ss), C.c_size_t(len(ss)), d, _p8(out), threads, lean)
        if rc:
            raise ValueError(f"oracle rc={rc}")
        return out

    def kmac_xof(self, k: bytes, x: bytes, l_bits: int, s: bytes, d: int) -> bytes:
        kd, ko = pack([k])
        xd, xo = pack([x])
        return self.kmac_xof_batch(kd, ko, xd, xo, l_bits, s, d)[0].tobytes()

    def cshake(self, x: bytes, l_bits: int, n: bytes, s: bytes, d: int) -> bytes:
        xd, xo = pack([x])
        return self.cshake_batch(xd, xo, l_bits, n, s, d)[0].tobytes()

    # ---- Ed448 side ----
    def fixed_base_batch(self, scalars_be56, threads=1):
        sc = _u8(scalars_be56)
        n = len(sc) // 56
        out = np.zeros((n, 112), dtype=np.uint8)
        self.lib.capy_ref_ed448_fixed_base_batch(_p8(sc), C.c_uint64(n), _p8(out), threads)
        return out

    def var_base_batch(self, scalars_be56, pts_xy112, threads=1):
        sc, pts = _u8(scalars_be56), _u8(pts_xy112)
        n = len(sc) // 56
        out = np.zeros((n, 112), dtype=np.uint8)
        rc = self.lib.capy_ref_ed448_var_base_batch(_p8(sc), _p8(pts), C.c_uint64(n), _p8(out), threads)
        return rc, out

    def keygen_batch(self, pws, pw_off, d, threads=1):
        pws, pw_off = _u8(pws), np.ascontiguousarray(pw_off, dtype=np.uint64)
        n = len(pw_off) - 1
        out = np.zeros((n, 112), dtype=np.uint8)
        rc = self.lib.capy_ref_ed448_keygen_batch(_p8(pws), _p64(pw_off), C.c_uint64(n), d, _p8(out), threads)
        if rc:
            raise ValueError(f"oracle rc={rc}")
        return out

    def sign_batch(self, pws, pw_off, msgs, msg_off, d, threads=1):
        pws, pw_off = _u8(pws), np.ascontiguousarray(pw_off, dtype=np.uint64)
        msgs, msg_off = _u8(msgs), np.ascontiguousarray(msg_off, dtype=np.uint64)
        n = len(pw_off) - 1
        h = np.zeros((n, 56), dtype=np.uint8)
        z = np.zeros((n, 56), dtype=np.uint8)
        rc = self.lib.capy_ref_ed448_sign_batch(_p8(pws), _p64(pw_off), _p8(msgs), _p64(msg_off), C.c_uint64(n), d,
                                                _p8(h), _p8(z), threads)
        if rc:
            raise ValueError(f"oracle rc={rc}")
        return h, z

    def verify_batch(self, pub_xy, msgs, msg_off, h, z, d, threads=1):
        pub, msgs, msg_off = _u8(pub_xy), _u8(msgs), np.ascontiguousarray(msg_off, dtype=np.uint64)
        h, z = _u8(h), _u8(z)
        n = len(msg_off) - 1
        ok = np.zeros(n, dtype=np.uint8)
        rc = self.lib.capy_ref_ed448_verify_batch(_p8(pub), _p8(msgs), _p64(msg_off), _p8(h), _p8(z), C.c_uint64(n), d,
                                                  _p8(ok), threads)
        if rc:
            raise ValueError(f"oracle rc={rc}")
        return ok

    def ecdh_batch(self, k_rand56, pub_xy, threads=1):
        k, pub = _u8(k_rand56), _u8(pub_xy)
        n = len(k) // 56
        out = np.zeros((n, 56), dtype=np.uint8)
        rc = self.lib.capy_ref_ed448_ecdh_batch(_p8(k), _p8(pub), C.c_uint64(n), _p8(out), threads)
        return rc, out

    def sc_mul_mod(self, a: bytes, b: bytes) -> bytes:
        o = np.zeros(56, np.uint8)
        self.lib.capy_ref_sc_mul_mod(_p8(_u8(a)), _p8(_u8(b)), _p8(o))
        return o.tobytes()

    def fe_mul(self, a: bytes, b: bytes) -> bytes:
        o = np.zeros(56, np.uint8)
        self.lib.capy_ref_fe_mul(_p8(_u8(a)), _p8(_u8(b)), _p8(o))
        return o.tobytes()

    def fe_inv(self, a: bytes) -> bytes:
        o = np.zeros(56, np.uint8)
        self.lib.capy_ref_fe_inv(_p8(_u8(a)), _p8(o))
        return o.tobytes()


_ORACLE = None


def get(native: bool = False) -> Oracle:
    global _ORACLE
    if native:
        return Oracle(native=True)
    if _ORACLE is None:
        _ORACLE = Oracle()
    return _ORACLE
