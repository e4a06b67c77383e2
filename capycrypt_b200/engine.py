"""Array-level Python front end of the C ABI (host numpy buffers and device torch tensors).

This is harness/plumbing: every function forwards to one C entry point of
libcapycrypt_gpu.so (include/capy_gpu.h).  torch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _binding as B


def _u8(a) -> np.ndarray:
    if isinstance(a, np.ndarray):
        return np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    b = bytes(a)
    return np.frombuffer(b, dtype=np.uint8).copy() if b else np.zeros(0, np.uint8)


def _u64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint64).reshape(-1)


def _hp(a: np.ndarray | None):
    """host address of a numpy buffer (a 1-byte dummy for empty arrays so it is never NULL)."""
    if a is None:
        return None
    if a.size == 0:
        return _DUMMY.ctypes.data
    return a.ctypes.data


_DUMMY = np.zeros(16, np.uint8)


def _out(out, shape, what: str) -> np.ndarray:
    """result buffer: a fresh (pageable) array, or the caller's -- e.g. pinned memory from Engine.pinned(), which the
    device-to-host copy then reaches at link speed."""
    if out is None:
        return np.zeros(shape, dtype=np.uint8)
    if not (isinstance(out, np.ndarray) and out.dtype == np.uint8 and out.flags.c_contiguous and out.flags.writeable):
        raise ValueError(f"{what}: out must be a writable C-contiguous uint8 array")
    _need(out.reshape(-1), int(np.prod(shape)), what)
    return out


def _need(buf: np.ndarray, nbytes: int, what: str) -> None:
    """The C side trusts (pointer, n): refuse a buffer shorter than n * stride here instead of letting the
    library read past a numpy allocation."""
    if buf.size < nbytes:
        raise ValueError(f"{what}: {buf.size} bytes, need {nbytes}")


def _need_packed(data: np.ndarray, off: np.ndarray, what: str) -> int:
    """packed batch = bytes + offsets[n + 1]: offsets start inside the buffer, never decrease, end inside it."""
    if off.size < 1:
        raise ValueError(f"{what}: offsets need n + 1 entries")
    if off.size > 1 and bool(np.any(off[1:] < off[:-1])):
        raise ValueError(f"{what}: offsets must not decrease")
    _need(data, int(off[-1]), what)
    return int(off.size) - 1


def pack(items) -> tuple[np.ndarray, np.ndarray]:
    """list of bytes-like -> (packed u8, u64 offsets[n+1])."""
    off = np.zeros(len(items) + 1, dtype=np.uint64)
    if len(items):
        off[1:] = np.cumsum([len(x) for x in items], dtype=np.uint64)
    blob = b"".join(bytes(x) for x in items)
    data = np.frombuffer(blob, dtype=np.uint8).copy() if blob else np.zeros(0, np.uint8)
    return data, off


class PreparedPublicKey:
    """A public key prepared on every device of one Engine (Engine.ed448_pub_prepare): the comb table of V that the
    engine's *_prepared calls use.  Reuse it across calls; close() it (or leave the `with` block) before the engine."""

    def __init__(self, engine: "Engine", handle: C.c_void_p, pub_xy112: bytes):
        self._engine = engine
        self.handle = handle
        self.pub_xy112 = pub_xy112

    @property
    def uses_comb(self) -> bool:
        """False when V has a torsion component: the prepared calls then run the variable-base pipelines"""
        return self._engine.lib.capy_ed448_pub_uses_comb(self.handle) == 1

    def close(self):
        if self.handle is not None and self.handle.value:
            self._engine.lib.capy_ed448_pub_free(self.handle)
        self.handle = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Hasher:
    """A batch of n resumable SHA3-d or KMACXOF streams on one Engine (Engine.sha3_hasher / Engine.kmac_xof_hasher).
    update() appends one piece per stream; final() returns what Engine.sha3 / Engine.kmac_xof return for the concatenated
    pieces.  close() it (or leave the `with` block) before the engine."""

    def __init__(self, engine: "Engine", handle: C.c_void_p, n: int, d: int, kmac: bool):
        self._engine = engine
        self.handle = handle
        self.n = n
        self.d = d
        self.kmac = kmac

    def device_range(self, dev_index: int = 0) -> tuple[int, int]:
        """the items [i0, i1) that live on device dev_index of the engine"""
        i0, i1 = C.c_uint64(0), C.c_uint64(0)
        self._engine._check(self._engine.lib.capy_hasher_device_range(self.handle, dev_index, C.byref(i0), C.byref(i1)))
        return int(i0.value), int(i1.value)

    def update(self, data, off) -> None:
        """capy_hasher_update: stream i appends data[off[i] .. off[i+1]) (blocking)"""
        data, off = _u8(data), _u64(off)
        if _need_packed(data, off, "hasher pieces") != self.n:
            raise ValueError(f"hasher update: {off.size - 1} pieces for {self.n} streams")
        self._engine._check(self._engine.lib.capy_hasher_update(self._engine._ctx, self.handle, _hp(data), _hp(off)))

    def final(self, out_bits: int | None = None, out_off=None, out: np.ndarray | None = None) -> np.ndarray:
        """capy_hasher_final: SHA3-d -> n x d/8 digests; KMACXOF -> n x out_bits/8, or packed by out_off"""
        out_bits = self.d if out_bits is None else out_bits
        if out_off is None:
            out = _out(out, (self.n, out_bits // 8), "hasher output")
            oo = None
        else:
            out_off = _u64(out_off)
            if out_off.size != self.n + 1 or bool(np.any(out_off[1:] < out_off[:-1])):
                raise ValueError("hasher final: out_off needs n + 1 non-decreasing entries")
            out = _out(out, (int(out_off[-1]),), "hasher output")
            oo = _hp(out_off)
        self._engine._check(self._engine.lib.capy_hasher_final(self._engine._ctx, self.handle, out_bits, oo, _hp(out)))
        return out

    def update_dev(self, t_data, t_off, dev_index: int = 0) -> None:
        """capy_hasher_update_dev on torch's current stream: t_off holds i1 - i0 + 1 offsets (device_range)"""
        self._engine._check(self._engine.lib.capy_hasher_update_dev(self._engine._ctx, self.handle, dev_index,
                                                                    self._engine._stream(), t_data.data_ptr(),
                                                                    t_off.data_ptr()))

    def final_dev(self, t_out, out_bits: int | None = None, t_out_off=None, dev_index: int = 0):
        """capy_hasher_final_dev on torch's current stream (the items of device_range(dev_index))"""
        out_bits = self.d if out_bits is None else out_bits
        self._engine._check(self._engine.lib.capy_hasher_final_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(), out_bits,
            t_out_off.data_ptr() if t_out_off is not None else None, t_out.data_ptr()))
        return t_out

    def export(self) -> np.ndarray:
        """capy_hasher_export: the streams as a blob (capy_gpu.h: the blob format; a KMACXOF blob is as secret as its
        keys), to be resumed by Engine.import_hasher in this or another engine (blocking)"""
        size = C.c_uint64(0)
        self._engine._check(self._engine.lib.capy_hasher_export_size(self.handle, C.byref(size)))
        blob = np.zeros(int(size.value), np.uint8)
        self._engine._check(self._engine.lib.capy_hasher_export(self._engine._ctx, self.handle, _hp(blob), blob.size))
        return blob

    def fork(self, src) -> "Hasher":
        """capy_hasher_fork: a new hasher of len(src) streams on the same engine; stream j starts as a copy of stream
        src[j] of this one, which is unchanged (blocking)"""
        src = _u64(src)
        h = C.c_void_p()
        self._engine._check(self._engine.lib.capy_hasher_fork(self._engine._ctx, self.handle, _hp(src), src.size,
                                                              C.byref(h)))
        return Hasher(self._engine, h, int(src.size), self.d, self.kmac)

    def close(self):
        if self.handle is not None and self.handle.value:
            self._engine.lib.capy_hasher_free(self.handle)
        self.handle = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EncryptStream(Hasher):
    """n seal streams (Engine.sponge_encrypt_stream / Engine.ed448_key_encrypt_stream): update() encrypts one piece per
    stream, final() returns the tags.  The concatenated ciphertext pieces and the tags are what the one-shot call gives
    for the concatenated plaintext."""

    def __init__(self, engine: "Engine", handle: C.c_void_p, n: int, d: int, tag_bytes: int):
        super().__init__(engine, handle, n, d, True)
        self.tag_bytes = tag_bytes

    def update(self, data, off, out: np.ndarray | None = None) -> np.ndarray:
        """capy_hasher_encrypt_update: the ciphertext of data[off[i] .. off[i+1]) at the same offsets of the result
        (out may be data itself: in place)"""
        data, off = _u8(data), _u64(off)
        if _need_packed(data, off, "stream pieces") != self.n:
            raise ValueError(f"stream update: {off.size - 1} pieces for {self.n} streams")
        out = _out(out, (data.size,), "stream ciphertext")
        self._engine._check(self._engine.lib.capy_hasher_encrypt_update(self._engine._ctx, self.handle, _hp(data), _hp(off),
                                                                        _hp(out)))
        return out

    def final(self, out: np.ndarray | None = None) -> np.ndarray:
        """the tags, n x tag_bytes"""
        return super().final(8 * self.tag_bytes, None, out)

    def update_dev(self, t_data, t_off, t_ct, dev_index: int = 0) -> None:
        """capy_hasher_encrypt_update_dev on torch's current stream (t_ct may be t_data)"""
        self._engine._check(self._engine.lib.capy_hasher_encrypt_update_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(), t_data.data_ptr(), t_off.data_ptr(),
            t_ct.data_ptr()))

    def final_dev(self, t_out, dev_index: int = 0):
        return super().final_dev(t_out, 8 * self.tag_bytes, None, dev_index)


class VerifyStream(Hasher):
    """n signature checks whose messages arrive in pieces (Engine.ed448_verify_stream): update() as Hasher, final()
    -> (rc, ok) as Engine.ed448_verify."""

    def __init__(self, engine: "Engine", handle: C.c_void_p, n: int, d: int):
        super().__init__(engine, handle, n, d, True)

    def final(self, ok_out: np.ndarray | None = None) -> tuple[int, np.ndarray]:
        ok = _out(ok_out, (self.n,), "verify flags")
        rc = self._engine._check(self._engine.lib.capy_hasher_verify_final(self._engine._ctx, self.handle, _hp(ok)),
                                 allow=(B.ERR_BAD_POINT,))
        return rc, ok

    def final_dev(self, t_ok, t_bad=None, dev_index: int = 0):
        """capy_hasher_verify_final_dev on torch's current stream; t_bad (one int32) gets 1 when a key was off the curve"""
        self._engine._check(self._engine.lib.capy_hasher_verify_final_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(), t_ok.data_ptr(),
            t_bad.data_ptr() if t_bad is not None else None))
        return t_ok


class SignStream(Hasher):
    """n signatures whose messages are fed twice (Engine.ed448_sign_stream): update() as Hasher in both passes,
    next_pass() between them, final() -> (h, z, ok).  ok[i] = 0: pass 2 carried other bytes than pass 1, and h[i], z[i]
    are zero."""

    def __init__(self, engine: "Engine", handle: C.c_void_p, n: int, d: int):
        super().__init__(engine, handle, n, d, True)

    def next_pass(self) -> None:
        """capy_hasher_next_pass (blocking)"""
        self._engine._check(self._engine.lib.capy_hasher_next_pass(self._engine._ctx, self.handle, None))

    def final(self) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        h, z = np.zeros((self.n, 56), dtype=np.uint8), np.zeros((self.n, 56), dtype=np.uint8)
        ok = np.zeros(self.n, dtype=np.uint8)
        self._engine._check(self._engine.lib.capy_hasher_sign_final(self._engine._ctx, self.handle, _hp(h), _hp(z), _hp(ok)))
        return h, z, ok

    def next_pass_dev(self, dev_index: int = 0) -> None:
        self._engine._check(self._engine.lib.capy_hasher_next_pass_dev(self._engine._ctx, self.handle, dev_index,
                                                                       self._engine._stream(), None, None))

    def final_dev(self, t_h, t_z, t_ok, dev_index: int = 0):
        """capy_hasher_sign_final_dev on torch's current stream"""
        self._engine._check(self._engine.lib.capy_hasher_sign_final_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(), t_h.data_ptr(), t_z.data_ptr(),
            t_ok.data_ptr()))


class DecryptStream(Hasher):
    """n decryptions whose ciphertexts are fed twice (Engine.sponge_decrypt_stream / Engine.ed448_key_decrypt_stream):
    update() takes the ciphertext in pass 1 and writes nothing, next_pass() -> (rc, verdicts), decrypt() takes the same
    ciphertext in pass 2 (plaintext out where the verdict was 1, the ciphertext elsewhere), final() -> (rc, ok).  rc is
    CAPY_OK or, for key_decrypt with an off-curve Z, ERR_BAD_POINT."""

    def __init__(self, engine: "Engine", handle: C.c_void_p, n: int, d: int):
        super().__init__(engine, handle, n, d, True)

    def next_pass(self, ok_out: np.ndarray | None = None) -> tuple[int, np.ndarray]:
        ok = _out(ok_out, (self.n,), "verdicts")
        rc = self._engine._check(self._engine.lib.capy_hasher_next_pass(self._engine._ctx, self.handle, _hp(ok)),
                                 allow=(B.ERR_BAD_POINT,))
        return rc, ok

    def decrypt(self, data, off, out: np.ndarray | None = None) -> np.ndarray:
        """capy_hasher_decrypt_update (out may be data itself: in place)"""
        data, off = _u8(data), _u64(off)
        if _need_packed(data, off, "stream pieces") != self.n:
            raise ValueError(f"stream decrypt: {off.size - 1} pieces for {self.n} streams")
        out = _out(out, (data.size,), "stream plaintext")
        self._engine._check(self._engine.lib.capy_hasher_decrypt_update(self._engine._ctx, self.handle, _hp(data), _hp(off),
                                                                        _hp(out)))
        return out

    def final(self, ok_out: np.ndarray | None = None) -> tuple[int, np.ndarray]:
        ok = _out(ok_out, (self.n,), "decrypt flags")
        rc = self._engine._check(self._engine.lib.capy_hasher_decrypt_final(self._engine._ctx, self.handle, _hp(ok)),
                                 allow=(B.ERR_BAD_POINT,))
        return rc, ok

    def next_pass_dev(self, t_ok=None, t_bad=None, dev_index: int = 0) -> None:
        self._engine._check(self._engine.lib.capy_hasher_next_pass_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(),
            t_ok.data_ptr() if t_ok is not None else None, t_bad.data_ptr() if t_bad is not None else None))

    def decrypt_dev(self, t_ct, t_off, t_out, dev_index: int = 0) -> None:
        """capy_hasher_decrypt_update_dev on torch's current stream (t_out may be t_ct)"""
        self._engine._check(self._engine.lib.capy_hasher_decrypt_update_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(), t_ct.data_ptr(), t_off.data_ptr(),
            t_out.data_ptr()))

    def final_dev(self, t_ok, t_bad=None, dev_index: int = 0):
        self._engine._check(self._engine.lib.capy_hasher_decrypt_final_dev(
            self._engine._ctx, self.handle, dev_index, self._engine._stream(), t_ok.data_ptr(),
            t_bad.data_ptr() if t_bad is not None else None))
        return t_ok


def hasher_blob_info(blob, lib=None) -> tuple[int, int, int]:
    """capy_hasher_blob_info (no GPU): (kind, d, n) of a blob from Hasher.export; kind 0 = SHA3-d, 1 = KMACXOF.
    CapyError(ERR_BAD_ARG) for a malformed header or a length that does not match it."""
    blob = _u8(blob)
    lib = lib or B.load()
    kind, d, n = C.c_int(0), C.c_int(0), C.c_uint64(0)
    rc = lib.capy_hasher_blob_info(_hp(blob), blob.size, C.byref(kind), C.byref(d), C.byref(n))
    if rc != B.OK:
        raise B.CapyError(rc, lib.capy_strerror(rc).decode())
    return int(kind.value), int(d.value), int(n.value)


def _pub_or_key(pub):
    """(pub_xy112 bytes or None, prepared key handle or None) of a PreparedPublicKey or n x 112 key bytes"""
    if isinstance(pub, PreparedPublicKey):
        return None, pub.handle
    return _u8(pub), None


class Engine:
    """One capy_ctx.  devices=None -> current CUDA device."""

    def __init__(self, devices=None):
        self.lib = B.load()
        self._ctx = C.c_void_p()
        self._pinned = []
        if devices is None:
            rc = self.lib.capy_gpu_init(None, 0, C.byref(self._ctx))
        else:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.lib.capy_gpu_init(arr, len(devices), C.byref(self._ctx))
        if rc != B.OK:
            self._ctx = C.c_void_p()
            raise B.CapyError(rc, self.lib.capy_strerror(rc).decode())

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            for p in self._pinned:
                self.lib.capy_host_free(p)
            self._pinned = []
            self.lib.capy_gpu_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def scrub(self):
        """zero every device scratch buffer of the ctx (intermediate secrets of the pipelines live there)"""
        self._check(self.lib.capy_gpu_scrub(self._ctx))

    def copy_probe(self, h_in: np.ndarray, h_out: np.ndarray, reps: int = 10, dev_index: int = 0) -> float:
        """capy_copy_probe: ms per repetition of (H2D of h_in) overlapped with (D2H into h_out), no kernel"""
        ms = C.c_double(0.0)
        self._check(self.lib.capy_copy_probe(self._ctx, dev_index, _hp(h_in), h_in.size, _hp(h_out), h_out.size, reps,
                                             C.byref(ms)))
        return float(ms.value)

    def set_plan_cache(self, enable: bool = True):
        """capy_gpu_set_plan_cache: ragged calls that pass the same offsets array again launch without a host round trip"""
        self._check(self.lib.capy_gpu_set_plan_cache(self._ctx, 1 if enable else 0))

    # ---- plumbing ----
    def _check(self, rc: int, allow=()):
        if rc != B.OK and rc not in allow:
            msg = self.lib.capy_strerror(rc).decode()
            if rc == B.ERR_CUDA:
                msg += " -- " + self.lib.capy_last_cuda_error(self._ctx).decode()
            raise B.CapyError(rc, msg)
        return rc

    @property
    def device_count(self) -> int:
        return self.lib.capy_gpu_device_count(self._ctx)

    @property
    def launch_count(self) -> int:
        return int(self.lib.capy_launch_count(self._ctx))

    def pinned(self, nbytes: int) -> np.ndarray:
        """uint8 numpy view of pinned host memory (capy_host_alloc); freed by close()."""
        p = self.lib.capy_host_alloc(max(nbytes, 1))
        if not p:
            raise MemoryError("capy_host_alloc failed")
        self._pinned.append(p)
        return np.ctypeslib.as_array((C.c_uint8 * max(nbytes, 1)).from_address(p))[:nbytes]

    # =================================================================================
    # host-buffer API (blocking)
    # =================================================================================
    def sha3(self, data, off, d: int, out: np.ndarray | None = None) -> np.ndarray:
        data, off = _u8(data), _u64(off)
        n = _need_packed(data, off, "sha3 messages")
        out = _out(out, (n, max(d // 8, 0) if d in (224, 256, 384, 512) else 1), "sha3 digests")
        self._check(self.lib.capy_sha3_batch(self._ctx, d, _hp(data), _hp(off), n, _hp(out), 0))
        return out

    def sha3_fixed(self, data, msg_len: int, stride: int, n: int, d: int, out: np.ndarray | None = None) -> np.ndarray:
        data = _u8(data)
        if n:
            _need(data, (n - 1) * stride + msg_len, "sha3_fixed messages")
        if out is None:
            out = np.zeros((n, d // 8 if d in (224, 256, 384, 512) else 1), dtype=np.uint8)
        elif d in (224, 256, 384, 512):
            _need(out.reshape(-1), n * (d // 8), "sha3_fixed digests")
        self._check(self.lib.capy_sha3_batch_fixed(self._ctx, d, _hp(data), msg_len, stride, n, _hp(out), 0))
        return out

    def cshake(self, data, off, out_bits: int, fn: bytes, custom: bytes, d: int, out: np.ndarray | None = None) -> np.ndarray:
        data, off = _u8(data), _u64(off)
        n = _need_packed(data, off, "cshake messages")
        out = _out(out, (n, out_bits // 8), "cshake output")
        fn_a, cs_a = _u8(fn), _u8(custom)
        self._check(self.lib.capy_cshake_batch(self._ctx, d, _hp(data), _hp(off), n, _hp(fn_a), len(fn_a), _hp(cs_a),
                                               len(cs_a), out_bits, _hp(out)))
        return out

    def kmac_xof(self, keys, key_off, data, off, out_bits: int, custom: bytes, d: int, out_off=None,
                 out: np.ndarray | None = None) -> np.ndarray:
        keys, key_off, data, off = _u8(keys), _u64(key_off), _u8(data), _u64(off)
        n = _need_packed(data, off, "kmac messages")
        if _need_packed(keys, key_off, "kmac keys") != n:
            raise ValueError("kmac: keys and messages differ in count")
        cs_a = _u8(custom)
        if out_off is None:
            out = _out(out, (n, out_bits // 8), "kmac output")
            oo = None
        else:
            out_off = _u64(out_off)
            if out_off.size != n + 1 or bool(np.any(out_off[1:] < out_off[:-1])):
                raise ValueError("kmac: out_off needs n + 1 non-decreasing entries")
            out = _out(out, (int(out_off[-1]),), "kmac output")
            oo = _hp(out_off)
        self._check(self.lib.capy_kmac_xof_batch(self._ctx, d, _hp(keys), _hp(key_off), _hp(data), _hp(off), n,
                                                 _hp(cs_a), len(cs_a), out_bits, oo, _hp(out)))
        return out

    def sha3_hasher(self, n: int, d: int) -> Hasher:
        """capy_sha3_hasher_new: n resumable SHA3-d streams (blocking)"""
        h = C.c_void_p()
        self._check(self.lib.capy_sha3_hasher_new(self._ctx, d, n, C.byref(h)))
        return Hasher(self, h, n, d, False)

    def kmac_xof_hasher(self, keys, key_off, custom: bytes, d: int) -> Hasher:
        """capy_kmac_xof_hasher_new: one resumable KMACXOF stream per key, customisation string `custom` (blocking)"""
        keys, key_off = _u8(keys), _u64(key_off)
        n = _need_packed(keys, key_off, "hasher keys")
        cs_a = _u8(custom)
        h = C.c_void_p()
        self._check(self.lib.capy_kmac_xof_hasher_new(self._ctx, d, _hp(keys), _hp(key_off), n, _hp(cs_a), len(cs_a),
                                                      C.byref(h)))
        return Hasher(self, h, n, d, True)

    def import_hasher(self, blob) -> Hasher:
        """capy_hasher_import: the streams of a blob from Hasher.export, dealt over this engine's devices (blocking)"""
        blob = _u8(blob)
        kind, d, n = hasher_blob_info(blob, self.lib)
        h = C.c_void_p()
        self._check(self.lib.capy_hasher_import(self._ctx, _hp(blob), blob.size, C.byref(h)))
        return Hasher(self, h, n, d, kind == 1)

    def sponge_encrypt_stream(self, pws, pw_off, nonces, nonce_len: int, d: int, variant: int = B.AE_SHA3) -> EncryptStream:
        """capy_sponge_encrypt_stream_new: one seal stream per password (blocking); tags of 64 bytes"""
        pws, pw_off, nonces = _u8(pws), _u64(pw_off), _u8(nonces)
        n = _need_packed(pws, pw_off, "stream passwords")
        if len(nonces) != n * nonce_len:
            raise ValueError(f"sponge_encrypt_stream: need {n} x {nonce_len} nonce bytes")
        h = C.c_void_p()
        self._check(self.lib.capy_sponge_encrypt_stream_new(self._ctx, d, variant, _hp(pws), _hp(pw_off), _hp(nonces),
                                                            nonce_len, n, C.byref(h)))
        return EncryptStream(self, h, n, d, 64)

    def ed448_key_encrypt_stream(self, pub, k_rand56, d: int) -> tuple[EncryptStream, np.ndarray]:
        """capy_ed448_key_encrypt_stream_new against n x 112 key bytes or a PreparedPublicKey (blocking) -> (streams with
        tags of 56 bytes, nonce points Z n x 112).  CapyError(ERR_BAD_POINT) for an off-curve key."""
        pub_b, key = _pub_or_key(pub)
        k = _u8(k_rand56)
        n = len(k) // 56
        if len(k) != n * 56 or (pub_b is not None and len(pub_b) != n * 112):
            raise ValueError(f"key_encrypt_stream: k holds {len(k)} bytes, need n x 56 and n x 112 key bytes")
        z = np.zeros((n, 112), dtype=np.uint8)
        h = C.c_void_p()
        self._check(self.lib.capy_ed448_key_encrypt_stream_new(self._ctx, d, _hp(pub_b), key, _hp(k), n, _hp(z),
                                                               C.byref(h)))
        return EncryptStream(self, h, n, d, 56), z

    def ed448_verify_stream(self, pub, h56, z_be56, d: int) -> VerifyStream:
        """capy_ed448_verify_stream_new against n x 112 key bytes or a PreparedPublicKey (blocking)"""
        pub_b, key = _pub_or_key(pub)
        hb, zb = _u8(h56), _u8(z_be56)
        n = len(hb) // 56
        if len(hb) != n * 56 or len(zb) != n * 56 or (pub_b is not None and len(pub_b) != n * 112):
            raise ValueError(f"verify_stream: h/z hold {len(hb)}/{len(zb)} bytes, need n x 56 and n x 112 key bytes")
        h = C.c_void_p()
        self._check(self.lib.capy_ed448_verify_stream_new(self._ctx, d, _hp(pub_b), key, _hp(hb), _hp(zb), n, C.byref(h)))
        return VerifyStream(self, h, n, d)

    def ed448_sign_stream(self, pws, pw_off, d: int) -> SignStream:
        """capy_ed448_sign_stream_new: one sign stream per password (blocking)"""
        pws, pw_off = _u8(pws), _u64(pw_off)
        n = _need_packed(pws, pw_off, "stream passwords")
        h = C.c_void_p()
        self._check(self.lib.capy_ed448_sign_stream_new(self._ctx, d, _hp(pws), _hp(pw_off), n, C.byref(h)))
        return SignStream(self, h, n, d)

    def sponge_decrypt_stream(self, pws, pw_off, nonces, nonce_len: int, tags64, d: int,
                              variant: int = B.AE_SHA3) -> DecryptStream:
        """capy_sponge_decrypt_stream_new: one open stream per password, expected tags n x 64 (blocking)"""
        pws, pw_off, nonces, tags = _u8(pws), _u64(pw_off), _u8(nonces), _u8(tags64)
        n = _need_packed(pws, pw_off, "stream passwords")
        if len(nonces) != n * nonce_len or len(tags) != n * 64:
            raise ValueError(f"sponge_decrypt_stream: need {n} x {nonce_len} nonce bytes and {n} x 64 tag bytes")
        h = C.c_void_p()
        self._check(self.lib.capy_sponge_decrypt_stream_new(self._ctx, d, variant, _hp(pws), _hp(pw_off), _hp(nonces),
                                                            nonce_len, _hp(tags), n, C.byref(h)))
        return DecryptStream(self, h, n, d)

    def ed448_key_decrypt_stream(self, pws, pw_off, z_xy112, tags56, d: int) -> DecryptStream:
        """capy_ed448_key_decrypt_stream_new: one key_decrypt stream per password and Z, expected tags n x 56 (blocking)"""
        pws, pw_off, z, tags = _u8(pws), _u64(pw_off), _u8(z_xy112), _u8(tags56)
        n = _need_packed(pws, pw_off, "stream passwords")
        if len(z) != n * 112 or len(tags) != n * 56:
            raise ValueError(f"key_decrypt_stream: need {n} x 112 Z bytes and {n} x 56 tag bytes")
        h = C.c_void_p()
        self._check(self.lib.capy_ed448_key_decrypt_stream_new(self._ctx, d, _hp(pws), _hp(pw_off), _hp(z), _hp(tags), n,
                                                               C.byref(h)))
        return DecryptStream(self, h, n, d)

    def ed448_fixed_base(self, scalars_be56, out: np.ndarray | None = None) -> np.ndarray:
        sc = _u8(scalars_be56)
        n = len(sc) // 56
        _need(sc, n * 56, "scalars")
        if len(sc) != n * 56:
            raise ValueError("scalars: length is not a multiple of 56")
        if out is None:
            out = np.zeros((n, 112), dtype=np.uint8)
        else:
            _need(out.reshape(-1), n * 112, "fixed_base output")
        self._check(self.lib.capy_ed448_fixed_base_batch(self._ctx, _hp(sc), n, _hp(out)))
        return out

    def ed448_var_base(self, scalars_be56, points_xy112) -> tuple[int, np.ndarray]:
        sc, pts = _u8(scalars_be56), _u8(points_xy112)
        n = len(sc) // 56
        if len(sc) != n * 56 or len(pts) != n * 112:
            raise ValueError(f"var_base: {len(sc)} scalar bytes / {len(pts)} point bytes are not n x 56 / n x 112")
        out = np.zeros((n, 112), dtype=np.uint8)
        rc = self._check(self.lib.capy_ed448_var_base_batch(self._ctx, _hp(sc), _hp(pts), n, _hp(out)),
                         allow=(B.ERR_BAD_POINT,))
        return rc, out

    def ed448_keygen(self, pws, pw_off, d: int, out: np.ndarray | None = None) -> np.ndarray:
        pws, pw_off = _u8(pws), _u64(pw_off)
        n = _need_packed(pws, pw_off, "keygen passwords")
        out = _out(out, (n, 112), "keygen output")
        self._check(self.lib.capy_ed448_keygen_batch(self._ctx, d, _hp(pws), _hp(pw_off), n, _hp(out)))
        return out

    def ed448_sign(self, pws, pw_off, msgs, msg_off, d: int, h_out: np.ndarray | None = None,
                   z_out: np.ndarray | None = None) -> tuple[np.ndarray, np.ndarray]:
        pws, pw_off, msgs, msg_off = _u8(pws), _u64(pw_off), _u8(msgs), _u64(msg_off)
        n = _need_packed(pws, pw_off, "sign passwords")
        if _need_packed(msgs, msg_off, "sign messages") != n:
            raise ValueError("sign: passwords and messages differ in count")
        h = _out(h_out, (n, 56), "sign h")
        z = _out(z_out, (n, 56), "sign z")
        self._check(self.lib.capy_ed448_sign_batch(self._ctx, d, _hp(pws), _hp(pw_off), _hp(msgs), _hp(msg_off), n,
                                                   _hp(h), _hp(z)))
        return h, z

    def ed448_verify(self, pub_xy112, msgs, msg_off, h56, z_be56, d: int, ok_out: np.ndarray | None = None) -> tuple[int, np.ndarray]:
        pub, msgs, msg_off, h, z = _u8(pub_xy112), _u8(msgs), _u64(msg_off), _u8(h56), _u8(z_be56)
        n = _need_packed(msgs, msg_off, "verify messages")
        if len(pub) != n * 112 or len(h) != n * 56 or len(z) != n * 56:
            raise ValueError(f"verify: pub/h/z hold {len(pub)}/{len(h)}/{len(z)} bytes, need {n} x 112/56/56")
        ok = _out(ok_out, (n,), "verify flags")
        rc = self._check(self.lib.capy_ed448_verify_batch(self._ctx, d, _hp(pub), _hp(msgs), _hp(msg_off), _hp(h),
                                                          _hp(z), n, _hp(ok)), allow=(B.ERR_BAD_POINT,))
        return rc, ok

    def ed448_ecdh(self, k_rand56, pub_xy112, want_z: bool = True):
        k, pub = _u8(k_rand56), _u8(pub_xy112)
        n = len(k) // 56
        if len(k) != n * 56 or len(pub) != n * 112:
            raise ValueError(f"ecdh: {len(k)} nonce bytes / {len(pub)} key bytes are not n x 56 / n x 112")
        wx = np.zeros((n, 56), dtype=np.uint8)
        z = np.zeros((n, 112), dtype=np.uint8) if want_z else None
        rc = self._check(self.lib.capy_ed448_ecdh_batch(self._ctx, _hp(k), _hp(pub), n, _hp(wx), _hp(z)),
                         allow=(B.ERR_BAD_POINT,))
        return rc, wx, z

    def sponge_encrypt(self, pws, pw_off, nonces, nonce_len: int, msgs, msg_off, d: int, variant: int = B.AE_SHA3):
        """-> (ciphertext packed like msgs, tags n x 64)."""
        pws, pw_off, nonces, msgs, msg_off = _u8(pws), _u64(pw_off), _u8(nonces), _u8(msgs), _u64(msg_off)
        n = _need_packed(msgs, msg_off, "sponge_encrypt messages")
        if _need_packed(pws, pw_off, "sponge_encrypt passwords") != n or len(nonces) != n * nonce_len:
            raise ValueError(f"sponge_encrypt: need {n} passwords and {n} x {nonce_len} nonce bytes")
        ct = np.zeros(len(msgs), dtype=np.uint8)
        tag = np.zeros((n, 64), dtype=np.uint8)
        self._check(self.lib.capy_sponge_encrypt_batch(self._ctx, d, variant, _hp(pws), _hp(pw_off), _hp(nonces), nonce_len,
                                                       _hp(msgs), _hp(msg_off), n, _hp(ct), _hp(tag)))
        return ct, tag

    def sponge_decrypt(self, pws, pw_off, nonces, nonce_len: int, ct, ct_off, tags, d: int, variant: int = B.AE_SHA3):
        """-> (buffer packed like ct, ok n)."""
        pws, pw_off, nonces, ct, ct_off, tags = _u8(pws), _u64(pw_off), _u8(nonces), _u8(ct), _u64(ct_off), _u8(tags)
        n = _need_packed(ct, ct_off, "sponge_decrypt ciphertexts")
        if _need_packed(pws, pw_off, "sponge_decrypt passwords") != n or len(nonces) != n * nonce_len or len(tags) != n * 64:
            raise ValueError(f"sponge_decrypt: need {n} passwords, {n} x {nonce_len} nonce bytes and {n} x 64 tag bytes")
        out = np.zeros(len(ct), dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8)
        self._check(self.lib.capy_sponge_decrypt_batch(self._ctx, d, variant, _hp(pws), _hp(pw_off), _hp(nonces), nonce_len,
                                                       _hp(ct), _hp(ct_off), _hp(tags), n, _hp(out), _hp(ok)))
        return out, ok

    def ed448_key_encrypt(self, pub_xy112, k_rand56, msgs, msg_off, d: int):
        """-> (rc, ciphertext, tags n x 56, nonce points Z n x 112)."""
        pub, k, msgs, msg_off = _u8(pub_xy112), _u8(k_rand56), _u8(msgs), _u64(msg_off)
        n = _need_packed(msgs, msg_off, "key_encrypt messages")
        if len(pub) != n * 112 or len(k) != n * 56:
            raise ValueError(f"key_encrypt: pub/k hold {len(pub)}/{len(k)} bytes, need {n} x 112/56")
        ct = np.zeros(len(msgs), dtype=np.uint8)
        tag = np.zeros((n, 56), dtype=np.uint8)
        z = np.zeros((n, 112), dtype=np.uint8)
        rc = self._check(self.lib.capy_ed448_key_encrypt_batch(self._ctx, d, _hp(pub), _hp(k), _hp(msgs), _hp(msg_off), n,
                                                               _hp(ct), _hp(tag), _hp(z)), allow=(B.ERR_BAD_POINT,))
        return rc, ct, tag, z

    def ed448_pub_prepare(self, pub_xy112) -> PreparedPublicKey:
        """capy_ed448_pub_prepare (blocking); CapyError(ERR_BAD_POINT) for an off-curve point."""
        pub = _u8(pub_xy112)
        if len(pub) != 112:
            raise ValueError(f"pub_prepare: {len(pub)} bytes, need 112")
        h = C.c_void_p()
        self._check(self.lib.capy_ed448_pub_prepare(self._ctx, _hp(pub), C.byref(h)))
        return PreparedPublicKey(self, h, pub.tobytes())

    def ed448_verify_prepared(self, key: PreparedPublicKey, msgs, msg_off, h56, z_be56, d: int,
                              ok_out: np.ndarray | None = None) -> np.ndarray:
        """ed448_verify with every public key = the prepared one."""
        msgs, msg_off, h, z = _u8(msgs), _u64(msg_off), _u8(h56), _u8(z_be56)
        n = _need_packed(msgs, msg_off, "verify messages")
        if len(h) != n * 56 or len(z) != n * 56:
            raise ValueError(f"verify: h/z hold {len(h)}/{len(z)} bytes, need {n} x 56/56")
        ok = _out(ok_out, (n,), "verify flags")
        self._check(self.lib.capy_ed448_verify_prepared_batch(self._ctx, d, key.handle, _hp(msgs), _hp(msg_off), _hp(h),
                                                              _hp(z), n, _hp(ok)))
        return ok

    def ed448_key_encrypt_prepared(self, key: PreparedPublicKey, k_rand56, msgs, msg_off, d: int):
        """ed448_key_encrypt with every public key = the prepared one -> (ciphertext, tags n x 56, nonce points Z n x 112)."""
        k, msgs, msg_off = _u8(k_rand56), _u8(msgs), _u64(msg_off)
        n = _need_packed(msgs, msg_off, "key_encrypt messages")
        if len(k) != n * 56:
            raise ValueError(f"key_encrypt: k holds {len(k)} bytes, need {n} x 56")
        ct = np.zeros(len(msgs), dtype=np.uint8)
        tag = np.zeros((n, 56), dtype=np.uint8)
        z = np.zeros((n, 112), dtype=np.uint8)
        self._check(self.lib.capy_ed448_key_encrypt_prepared_batch(self._ctx, d, key.handle, _hp(k), _hp(msgs), _hp(msg_off),
                                                                   n, _hp(ct), _hp(tag), _hp(z)))
        return ct, tag, z

    def ed448_key_decrypt(self, pws, pw_off, z_xy112, ct, ct_off, tags, d: int):
        """-> (rc, buffer packed like ct, ok n)."""
        pws, pw_off, z, ct, ct_off, tags = _u8(pws), _u64(pw_off), _u8(z_xy112), _u8(ct), _u64(ct_off), _u8(tags)
        n = _need_packed(ct, ct_off, "key_decrypt ciphertexts")
        if _need_packed(pws, pw_off, "key_decrypt passwords") != n or len(z) != n * 112 or len(tags) != n * 56:
            raise ValueError(f"key_decrypt: need {n} passwords, {n} x 112 nonce-point bytes and {n} x 56 tag bytes")
        out = np.zeros(len(ct), dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8)
        rc = self._check(self.lib.capy_ed448_key_decrypt_batch(self._ctx, d, _hp(pws), _hp(pw_off), _hp(z), _hp(ct),
                                                               _hp(ct_off), _hp(tags), n, _hp(out), _hp(ok)),
                         allow=(B.ERR_BAD_POINT,))
        return rc, out, ok

    # =================================================================================
    # device-pointer API (async on torch's current stream); tensors are torch.uint8 / int64 CUDA
    # =================================================================================
    @staticmethod
    def _stream():
        import torch

        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def sha3_dev(self, t_data, t_off, d: int, t_out, dev_index: int = 0):
        n = t_off.numel() - 1
        self._check(self.lib.capy_sha3_batch_dev(self._ctx, dev_index, self._stream(), d, t_data.data_ptr(),
                                                 t_off.data_ptr(), n, t_out.data_ptr(), 0))
        return t_out

    def sha3_fixed_dev(self, t_data, msg_len: int, stride: int, n: int, d: int, t_out, dev_index: int = 0):
        self._check(self.lib.capy_sha3_batch_fixed_dev(self._ctx, dev_index, self._stream(), d, t_data.data_ptr(),
                                                       msg_len, stride, n, t_out.data_ptr(), 0))
        return t_out

    def cshake_dev(self, t_data, t_off, out_bits: int, fn: bytes, custom: bytes, d: int, t_out, dev_index: int = 0):
        n = t_off.numel() - 1
        fn_a, cs_a = _u8(fn), _u8(custom)
        self._check(self.lib.capy_cshake_batch_dev(self._ctx, dev_index, self._stream(), d, t_data.data_ptr(),
                                                   t_off.data_ptr(), n, _hp(fn_a), len(fn_a), _hp(cs_a), len(cs_a),
                                                   out_bits, t_out.data_ptr()))
        return t_out

    def kmac_xof_dev(self, t_keys, t_key_off, t_data, t_off, out_bits: int, custom: bytes, d: int, t_out,
                     t_out_off=None, dev_index: int = 0):
        n = t_off.numel() - 1
        cs_a = _u8(custom)
        self._check(self.lib.capy_kmac_xof_batch_dev(
            self._ctx, dev_index, self._stream(), d, t_keys.data_ptr(), t_key_off.data_ptr(), t_data.data_ptr(),
            t_off.data_ptr(), n, _hp(cs_a), len(cs_a), out_bits,
            t_out_off.data_ptr() if t_out_off is not None else None, t_out.data_ptr()))
        return t_out

    def kmac_xof_fixed_dev(self, t_keys, key_len: int, key_stride: int, t_data, msg_len: int, msg_stride: int, n: int,
                           out_bits: int, custom: bytes, d: int, t_out, dev_index: int = 0):
        cs_a = _u8(custom)
        self._check(self.lib.capy_kmac_xof_batch_fixed_dev(
            self._ctx, dev_index, self._stream(), d, t_keys.data_ptr(), key_len, key_stride,
            t_data.data_ptr() if t_data is not None else None, msg_len, msg_stride, n, _hp(cs_a), len(cs_a), out_bits,
            t_out.data_ptr()))
        return t_out

    def fips_shake_dev(self, t_data, t_off, shake_bits: int, out_bytes: int, t_out, dev_index: int = 0):
        n = t_off.numel() - 1
        self._check(self.lib.capy_fips_shake_batch_dev(self._ctx, dev_index, self._stream(), shake_bits,
                                                       t_data.data_ptr(), t_off.data_ptr(), n, out_bytes,
                                                       t_out.data_ptr()))
        return t_out

    def ed448_fixed_base_dev(self, t_scalars, n: int, t_out, dev_index: int = 0):
        self._check(self.lib.capy_ed448_fixed_base_batch_dev(self._ctx, dev_index, self._stream(),
                                                             t_scalars.data_ptr(), n, t_out.data_ptr()))
        return t_out

    def ed448_var_base_dev(self, t_scalars, t_points, n: int, t_out, t_bad=None, dev_index: int = 0):
        self._check(self.lib.capy_ed448_var_base_batch_dev(self._ctx, dev_index, self._stream(), t_scalars.data_ptr(),
                                                           t_points.data_ptr(), n, t_out.data_ptr(),
                                                           t_bad.data_ptr() if t_bad is not None else None))
        return t_out

    def ed448_keygen_dev(self, t_pws, t_pw_off, d: int, t_out, dev_index: int = 0):
        n = t_pw_off.numel() - 1
        self._check(self.lib.capy_ed448_keygen_batch_dev(self._ctx, dev_index, self._stream(), d, t_pws.data_ptr(),
                                                         t_pw_off.data_ptr(), n, t_out.data_ptr()))
        return t_out

    def ed448_sign_dev(self, t_pws, t_pw_off, t_msgs, t_msg_off, d: int, t_h, t_z, dev_index: int = 0):
        n = t_pw_off.numel() - 1
        self._check(self.lib.capy_ed448_sign_batch_dev(self._ctx, dev_index, self._stream(), d, t_pws.data_ptr(),
                                                       t_pw_off.data_ptr(), t_msgs.data_ptr(), t_msg_off.data_ptr(), n,
                                                       t_h.data_ptr(), t_z.data_ptr()))

    def ed448_verify_dev(self, t_pub, t_msgs, t_msg_off, t_h, t_z, d: int, t_ok, t_bad=None, dev_index: int = 0):
        n = t_msg_off.numel() - 1
        self._check(self.lib.capy_ed448_verify_batch_dev(self._ctx, dev_index, self._stream(), d, t_pub.data_ptr(),
                                                         t_msgs.data_ptr(), t_msg_off.data_ptr(), t_h.data_ptr(),
                                                         t_z.data_ptr(), n, t_ok.data_ptr(),
                                                         t_bad.data_ptr() if t_bad is not None else None))
        return t_ok

    def sponge_encrypt_dev(self, t_pws, t_pw_off, pw_bytes: int, t_nonces, nonce_len: int, t_msgs, t_msg_off, d: int, t_ct,
                           t_tag, variant: int = B.AE_SHA3, dev_index: int = 0):
        n = t_msg_off.numel() - 1
        self._check(self.lib.capy_sponge_encrypt_batch_dev(
            self._ctx, dev_index, self._stream(), d, variant, t_pws.data_ptr(), t_pw_off.data_ptr(), pw_bytes,
            t_nonces.data_ptr(), nonce_len, t_msgs.data_ptr(), t_msg_off.data_ptr(), n, t_ct.data_ptr(), t_tag.data_ptr()))

    def sponge_decrypt_dev(self, t_pws, t_pw_off, pw_bytes: int, t_nonces, nonce_len: int, t_ct, t_ct_off, t_tag, d: int,
                           t_out, t_ok, variant: int = B.AE_SHA3, dev_index: int = 0):
        n = t_ct_off.numel() - 1
        self._check(self.lib.capy_sponge_decrypt_batch_dev(
            self._ctx, dev_index, self._stream(), d, variant, t_pws.data_ptr(), t_pw_off.data_ptr(), pw_bytes,
            t_nonces.data_ptr(), nonce_len, t_ct.data_ptr(), t_ct_off.data_ptr(), t_tag.data_ptr(), n, t_out.data_ptr(),
            t_ok.data_ptr()))

    def ed448_key_encrypt_dev(self, t_pub, t_k, t_msgs, t_msg_off, d: int, t_ct, t_tag, t_z, t_bad=None, dev_index: int = 0):
        n = t_msg_off.numel() - 1
        self._check(self.lib.capy_ed448_key_encrypt_batch_dev(
            self._ctx, dev_index, self._stream(), d, t_pub.data_ptr(), t_k.data_ptr(), t_msgs.data_ptr(),
            t_msg_off.data_ptr(), n, t_ct.data_ptr(), t_tag.data_ptr(), t_z.data_ptr(),
            t_bad.data_ptr() if t_bad is not None else None))

    def ed448_key_decrypt_dev(self, t_pws, t_pw_off, t_z, t_ct, t_ct_off, t_tag, d: int, t_out, t_ok, t_bad=None,
                              dev_index: int = 0):
        n = t_ct_off.numel() - 1
        self._check(self.lib.capy_ed448_key_decrypt_batch_dev(
            self._ctx, dev_index, self._stream(), d, t_pws.data_ptr(), t_pw_off.data_ptr(), t_z.data_ptr(),
            t_ct.data_ptr(), t_ct_off.data_ptr(), t_tag.data_ptr(), n, t_out.data_ptr(), t_ok.data_ptr(),
            t_bad.data_ptr() if t_bad is not None else None))

    def ed448_verify_prepared_dev(self, key: PreparedPublicKey, t_msgs, t_msg_off, t_h, t_z, d: int, t_ok,
                                  dev_index: int = 0):
        n = t_msg_off.numel() - 1
        self._check(self.lib.capy_ed448_verify_prepared_batch_dev(self._ctx, dev_index, self._stream(), d, key.handle,
                                                                  t_msgs.data_ptr(), t_msg_off.data_ptr(), t_h.data_ptr(),
                                                                  t_z.data_ptr(), n, t_ok.data_ptr()))
        return t_ok

    def ed448_key_encrypt_prepared_dev(self, key: PreparedPublicKey, t_k, t_msgs, t_msg_off, d: int, t_ct, t_tag, t_z,
                                       dev_index: int = 0):
        n = t_msg_off.numel() - 1
        self._check(self.lib.capy_ed448_key_encrypt_prepared_batch_dev(
            self._ctx, dev_index, self._stream(), d, key.handle, t_k.data_ptr(), t_msgs.data_ptr(), t_msg_off.data_ptr(),
            n, t_ct.data_ptr(), t_tag.data_ptr(), t_z.data_ptr()))
