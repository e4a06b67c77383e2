"""GPU: resumable SHA3-d and KMACXOF streams (capy_*_hasher_*): messages fed in pieces give, byte for byte, what the
one-shot batch calls and the oracle give for the concatenated pieces."""
from __future__ import annotations

import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pytest

from capycrypt_b200 import _binding as B
from capycrypt_b200.engine import Engine, pack

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
SHA3_RATE = {224: 144, 256: 136, 384: 104, 512: 72}
KMAC_RATE = {256: 168, 384: 152, 512: 136}
Q3_KEYS = {256: (163, 331), 384: (147, 299), 512: (131, 267)}  # key lengths whose bytepad content is a multiple of w
TAG = b"My Tagged Application"


@pytest.fixture(scope="module")
def eng():
    import torch

    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    torch.cuda.set_device(0)
    e = Engine()
    yield e
    e.close()


@pytest.fixture(scope="module")
def kat():
    with open(os.path.join(HERE, "golden", "sha3_kat.json")) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def orc():
    from oracle import cpu

    return cpu.get()


# ---- inputs ---------------------------------------------------------------------------------------------------------
def lengths(rnd, n, r):
    """message lengths with the edge cases up front: empty, r - 1, r, r + 1, len % 136 == 135, 2 r - 1, 2 r"""
    edge = [0, r - 1, r, r + 1, 135, 271, 2 * r - 1, 2 * r, 1, 3 * r + 5]
    return [edge[i] if i < len(edge) else int(rnd.integers(0, 3 * r + 8)) for i in range(n)]


def chunking(rnd, length, r, updates):
    """`updates` piece lengths that add up to `length`: cuts at 1, r - 1, r, r + 1 when they fit, the rest seeded;
    the remaining pieces are empty, at seeded places"""
    cuts = {c for c in (1, r - 1, r, r + 1) if 0 < c < length}
    while len(cuts) < updates - 2 and len(cuts) < length - 1:
        cuts.add(int(rnd.integers(1, length)))
    cuts = sorted(cuts)[: updates - 1]
    bounds = [0] + cuts + [length]
    lens = [b - a for a, b in zip(bounds, bounds[1:])]
    while len(lens) < updates:
        lens.insert(int(rnd.integers(0, len(lens) + 1)), 0)
    return lens


def feed(h, msgs, rnd, r, updates):
    """feeds every message through h.update in `updates` calls; returns nothing"""
    plan = [chunking(rnd, len(m), r, updates) for m in msgs]
    pos = [0] * len(msgs)
    for k in range(updates):
        pieces = []
        for i, m in enumerate(msgs):
            pieces.append(m[pos[i]:pos[i] + plan[i][k]])
            pos[i] += plan[i][k]
        h.update(*pack(pieces))
    assert all(p == len(m) for p, m in zip(pos, msgs))


def kmac_keys(rnd, n, d):
    q = Q3_KEYS[d]
    edge = [b"", bytes(q[0]), bytes(range(256)) * 2, bytes(q[1])]
    edge = [e[:q[1]] if i == 2 else e for i, e in enumerate(edge)]
    return [edge[i] if i < len(edge) else rnd.bytes(int(rnd.integers(0, 80))) for i in range(n)]


# ---- 1. parity with the one-shot calls and the oracle ---------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [224, 256, 384, 512])
def test_sha3_parity(eng, orc, d, n):
    rnd = np.random.default_rng(d * 7 + n)
    r = SHA3_RATE[d]
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, r)]
    with eng.sha3_hasher(n, d) as h:
        feed(h, msgs, rnd, r, 6)
        got = h.final()
    data, off = pack(msgs)
    assert np.array_equal(got, eng.sha3(data, off, d))
    assert np.array_equal(got, orc.sha3_batch(data, off, d))


@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_kmac_parity(eng, orc, d, n):
    rnd = np.random.default_rng(d * 11 + n)
    r = KMAC_RATE[d]
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, r)]
    keys = kmac_keys(rnd, n, d)
    s = TAG if n in (127, 4099) else b""
    kd, ko = pack(keys)
    data, off = pack(msgs)
    with eng.kmac_xof_hasher(kd, ko, s, d) as h:
        feed(h, msgs, rnd, r, 5)
        if n == 4099:  # per-item output lengths, some empty
            oo = np.zeros(n + 1, np.uint64)
            oo[1:] = np.cumsum(rnd.integers(0, 300, size=n).astype(np.uint64))
            got = h.final(None, oo)
            want = eng.kmac_xof(kd, ko, data, off, 0, s, d, out_off=oo)
            assert np.array_equal(got, want)
            for i in range(0, n, 97):  # the oracle per item
                L = int(oo[i + 1] - oo[i])
                if L:
                    exp = orc.kmac_xof(keys[i], msgs[i], 8 * L, s, d)
                    assert got[int(oo[i]):int(oo[i + 1])].tobytes() == exp, i
            return
        bits = {1: 8, 127: d, 129: 4096}[n]
        got = h.final(bits)
    assert np.array_equal(got, eng.kmac_xof(kd, ko, data, off, bits, s, d))
    assert np.array_equal(got, orc.kmac_xof_batch(kd, ko, data, off, bits, s, d))


def test_api_streams(orc):
    from capycrypt_b200.api import Gpu, SecParam

    g = Gpu()
    with g.sha3_stream(2, SecParam.D256) as st:
        st.update([b"ab", b""])
        st.update([b"c" * 300, b"xyz"])
        assert st.finish() == [orc.sha3(b"ab" + b"c" * 300, 256), orc.sha3(b"xyz", 256)]
    with g.kmac_xof_stream([b"pw1", b"pw2"], "My Tagged Application", SecParam.D512) as st:
        st.update([b"hello ", b""])
        st.update([b"world", b"!"])
        assert st.finish(512) == [orc.kmac_xof(b"pw1", b"hello world", 512, TAG, 512),
                                  orc.kmac_xof(b"pw2", b"!", 512, TAG, 512)]
    with pytest.raises(ValueError):
        g.kmac_xof_stream([b"k"], "", SecParam.D224)
    g.engine.close()


# ---- 2. the reference's KATs, one byte per update -------------------------------------------------------------------
def test_kats_one_byte_per_update(eng, kat):
    for row in kat["sha3"]:
        msg = bytes.fromhex(row["msg"])
        with eng.sha3_hasher(1, row["d"]) as h:
            for b in msg:
                h.update(np.frombuffer(bytes([b]), np.uint8), np.array([0, 1], np.uint64))
            assert h.final()[0].tobytes().hex() == row["digest"], row
    rows = [(r["pw"], r["msg"], r["s"], r["d"], r["d"], r["digest"]) for r in kat["tagged_hash"]]
    rows += [(r["k"], r["x"], r["s"], r["l"], r["d"], r["out"]) for r in kat["kmac_xof"]]
    assert rows
    for k, x, s, l, d, want in rows:
        if d == 224:
            continue
        k, x, s = bytes.fromhex(k), bytes.fromhex(x), bytes.fromhex(s)
        with eng.kmac_xof_hasher(*pack([k]), s, d) as h:
            for b in x:
                h.update(np.frombuffer(bytes([b]), np.uint8), np.array([0, 1], np.uint64))
            h.update(np.zeros(0, np.uint8), np.array([0, 0], np.uint64))
            assert h.final(l)[0].tobytes().hex() == want, (d, l)


# ---- 3. _dev calls on guarded buffers --------------------------------------------------------------------------------
GUARD = 4096


class Guarded:
    def __init__(self, nbytes, offset, fill=None, seed=0):
        import torch

        self.lo = GUARD + offset
        self.hi = self.lo + nbytes
        host = np.random.default_rng(seed + 31 * offset + nbytes).integers(0, 256, size=self.hi + GUARD, dtype=np.uint8)
        if fill is not None:
            host[self.lo:self.hi] = np.frombuffer(bytes(fill), np.uint8)
        self.pattern = host
        self.buf = torch.from_numpy(host.copy()).cuda()

    @property
    def ptr(self):
        return self.buf.data_ptr() + self.lo

    def get(self):
        whole = self.buf.cpu().numpy()
        assert np.array_equal(whole[:self.lo], self.pattern[:self.lo]), "write below the buffer"
        assert np.array_equal(whole[self.hi:], self.pattern[self.hi:]), "write past the end of the buffer"
        return whole[self.lo:self.hi].copy()


class _Ptr:
    def __init__(self, p):
        self.p = p

    def data_ptr(self):
        return self.p


@pytest.mark.parametrize("offset", [0, 1])
@pytest.mark.parametrize("kind", ["sha3", "kmac"])
def test_dev_guarded(eng, orc, kind, offset):
    import torch

    n, d = 129, 512 if kind == "kmac" else 256
    r = KMAC_RATE[d] if kind == "kmac" else SHA3_RATE[d]
    rnd = np.random.default_rng(5 + offset)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, r)]
    plan = [chunking(rnd, len(m), r, 4) for m in msgs]
    keys = kmac_keys(rnd, n, 512)
    h = eng.kmac_xof_hasher(*pack(keys), TAG, d) if kind == "kmac" else eng.sha3_hasher(n, d)
    assert h.device_range(0) == (0, n)
    pos = [0] * n
    for k in range(4):
        pieces = []
        for i, m in enumerate(msgs):
            pieces.append(m[pos[i]:pos[i] + plan[i][k]])
            pos[i] += plan[i][k]
        data, off = pack(pieces)
        gd = Guarded(len(data), offset, data, seed=k)
        go = Guarded(8 * (n + 1), 8 * offset, off.tobytes(), seed=100 + k)
        h.update_dev(_Ptr(gd.ptr), _Ptr(go.ptr))
        torch.cuda.synchronize()
        gd.get()
        go.get()
    wd, wo = pack(msgs)
    if kind == "sha3":
        out = Guarded(n * 32, offset, seed=7)
        h.final_dev(_Ptr(out.ptr))
        got = out.get().reshape(n, 32)
        want = orc.sha3_batch(wd, wo, d)
    else:
        oo = np.zeros(n + 1, np.uint64)
        oo[1:] = np.cumsum(rnd.integers(1, 200, size=n).astype(np.uint64))
        goo = Guarded(8 * (n + 1), 8 * offset, oo.tobytes(), seed=9)
        out = Guarded(int(oo[-1]), offset, seed=8)
        h.final_dev(_Ptr(out.ptr), 0, _Ptr(goo.ptr))
        got = out.get()
        goo.get()
        kd, ko = pack(keys)
        want = eng.kmac_xof(kd, ko, wd, wo, 0, TAG, d, out_off=oo)
    torch.cuda.synchronize()
    assert np.array_equal(got, want)
    h.close()


# ---- 4. what launches -------------------------------------------------------------------------------------------------
def _kernels(fn, tmp_path):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    out = []
    for e in ev:
        if e.get("cat") == "kernel" and "capy::" in e.get("name", ""):
            s = e["name"].replace("void ", "").replace("capy::", "")
            out.append(re.sub(r"\((?:unsigned )?int\)", "", s).split("(", 1)[0].replace(" ", ""))
    return out


def test_launches(eng, tmp_path):
    rnd = np.random.default_rng(3)
    n = 300
    msgs = [rnd.bytes(int(x)) for x in rnd.integers(0, 700, size=n)]
    data, off = pack(msgs)
    box = {}
    s = b"launch test " + rnd.bytes(8)  # not in the prefix cache yet
    ks = _kernels(lambda: box.__setitem__("k", eng.kmac_xof_hasher(*pack([b"key"] * n), s, 256)), tmp_path)
    assert sorted(set(ks)) == ["prefix_state_kernel<21>", "sponge_chain_kernel<21>"], ks
    box["s"] = eng.sha3_hasher(n, 384)
    for h, L in ((box["k"], 21), (box["s"], 13)):
        ks = _kernels(lambda: (h.update(data, off), h.update(data, off)), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>"] * 2, ks
        ks = _kernels(lambda: h.final(), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>"], ks
        h.close()


# ---- 5. isolation from the one-shot calls ----------------------------------------------------------------------------
def test_isolation(eng, orc):
    rnd = np.random.default_rng(17)
    n = 1000
    r_s, r_k = SHA3_RATE[256], KMAC_RATE[512]
    ms = [rnd.bytes(L) for L in lengths(rnd, n, r_s)]
    mk = [rnd.bytes(L) for L in lengths(rnd, n, r_k)]
    keys = kmac_keys(rnd, n, 512)
    hs = eng.sha3_hasher(n, 256)
    hk = eng.kmac_xof_hasher(*pack(keys), TAG, 512)
    ps = [chunking(rnd, len(m), r_s, 4) for m in ms]
    pk = [chunking(rnd, len(m), r_k, 4) for m in mk]
    # one-shot batches large enough for the chain-cut and dependent-job launches (the chain scratch slots)
    big = 1 << 16
    bd = rnd.integers(0, 256, size=big * 2048, dtype=np.uint8)
    bo = np.arange(big + 1, dtype=np.uint64) * 2048
    bk, bko = pack([b"k" * 32] * big)
    pw, pwo = pack([b"pw"] * big)
    nonces = rnd.integers(0, 256, size=big * 16, dtype=np.uint8)
    mm = rnd.integers(0, 256, size=big * 64, dtype=np.uint8)
    mo = np.arange(big + 1, dtype=np.uint64) * 64
    ct, tags = eng.sponge_encrypt(pw, pwo, nonces, 16, mm, mo, 512)
    pos_s, pos_k = [0] * n, [0] * n
    for k in range(4):
        a = []
        for i, m in enumerate(ms):
            a.append(m[pos_s[i]:pos_s[i] + ps[i][k]])
            pos_s[i] += ps[i][k]
        hs.update(*pack(a))
        eng.sha3(bd, bo, 256)
        b = []
        for i, m in enumerate(mk):
            b.append(m[pos_k[i]:pos_k[i] + pk[i][k]])
            pos_k[i] += pk[i][k]
        hk.update(*pack(b))
        tk = eng.kmac_xof(bk, bko, bd, bo, 512, TAG, 512)
        out, ok = eng.sponge_decrypt(pw, pwo, nonces, 16, ct, mo, tags, 512)
        assert ok.all() and np.array_equal(out, mm)
    assert np.array_equal(tk[:3], orc.kmac_xof_batch(*pack([b"k" * 32] * 3), bd[:3 * 2048], bo[:4], 512, TAG, 512))
    assert np.array_equal(hs.final(), orc.sha3_batch(*pack(ms), 256))
    assert np.array_equal(hk.final(512), orc.kmac_xof_batch(*pack(keys), *pack(mk), 512, TAG, 512))
    hs.close()
    hk.close()


# ---- 6. errors ----------------------------------------------------------------------------------------------------------
def test_errors(eng):
    lib = eng.lib
    h = C.c_void_p()
    kd, ko = pack([b"k"])
    assert lib.capy_kmac_xof_hasher_new(eng._ctx, 224, kd.ctypes.data, ko.ctypes.data, 1, None, 0, C.byref(h)) == B.ERR_BAD_ARG
    assert not h.value
    assert lib.capy_kmac_xof_hasher_new(eng._ctx, 300, kd.ctypes.data, ko.ctypes.data, 1, None, 0, C.byref(h)) == B.ERR_BAD_SECPARAM
    assert lib.capy_sha3_hasher_new(eng._ctx, 100, 1, C.byref(h)) == B.ERR_BAD_SECPARAM
    lib.capy_hasher_free(None)
    with eng.sha3_hasher(2, 256) as hs:
        hs.update(*pack([b"a", b"b"]))
        with pytest.raises(B.CapyError) as e:
            hs.final(512)  # SHA3-d: out_bits == d_bits
        assert e.value.status == B.ERR_BAD_ARG
        hs.final()
        for call in (lambda: hs.update(*pack([b"a", b"b"])), lambda: hs.final()):
            with pytest.raises(B.CapyError) as e:
                call()
            assert e.value.status == B.ERR_BAD_ARG
    other = Engine()
    try:
        with eng.sha3_hasher(2, 256) as hs:
            d, o = pack([b"a", b"b"])
            assert lib.capy_hasher_update(other._ctx, hs.handle, d.ctypes.data, o.ctypes.data) == B.ERR_BAD_ARG
            out = np.zeros(64, np.uint8)
            assert lib.capy_hasher_final(other._ctx, hs.handle, 256, None, out.ctypes.data) == B.ERR_BAD_ARG
            assert lib.capy_hasher_update_dev(other._ctx, hs.handle, 0, None, d.ctypes.data, o.ctypes.data) == B.ERR_BAD_ARG
            assert lib.capy_hasher_final_dev(other._ctx, hs.handle, 0, None, 256, None, out.ctypes.data) == B.ERR_BAD_ARG
            hs.update(d, o)
            assert hs.final()[1].tobytes() == eng.sha3(*pack([b"b"]), 256)[0].tobytes()
    finally:
        other.close()
    with eng.sha3_hasher(0, 512) as h0:  # n == 0: calls do nothing
        h0.update(np.zeros(0, np.uint8), np.zeros(1, np.uint64))
        assert h0.final().shape == (0, 64)


# ---- 7. scale -------------------------------------------------------------------------------------------------------------
def test_scale_2e16_streams(eng, orc):
    import torch

    n, updates, piece = 1 << 16, 64, 4096
    idx = np.array(sorted(set(np.random.default_rng(1).choice(n, 200, replace=False).tolist())
                          | {0, n - 1} | set(range(128 * ((n - 1) // 128), n))))
    t_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * piece
    g = torch.Generator(device="cuda")
    g.manual_seed(11)
    kept = [bytearray() for _ in idx]
    ti = torch.from_numpy(idx).cuda()
    with eng.sha3_hasher(n, 256) as h:
        for _ in range(updates):
            t = torch.randint(0, 256, (n, piece), dtype=torch.uint8, device="cuda", generator=g)
            h.update_dev(t, t_off)
            rows = t.index_select(0, ti).cpu().numpy()
            for j in range(len(idx)):
                kept[j] += rows[j].tobytes()
        out = torch.zeros(n, 32, dtype=torch.uint8, device="cuda")
        h.final_dev(out)
        torch.cuda.synchronize()
    got = out.cpu().numpy()[idx]
    assert np.array_equal(got, orc.sha3_batch(*pack([bytes(k) for k in kept]), 256, threads=orc.max_threads))


# ---- 8. two devices ---------------------------------------------------------------------------------------------------------
def test_two_devices(orc):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    e2 = Engine([0, 1])
    try:
        rnd = np.random.default_rng(21)
        n = 301
        msgs = [rnd.bytes(L) for L in lengths(rnd, n, 136)]
        keys = kmac_keys(rnd, n, 512)
        h = e2.kmac_xof_hasher(*pack(keys), TAG, 512)
        (a0, a1), (b0, b1) = h.device_range(0), h.device_range(1)
        assert a0 == 0 and a1 == b0 and b1 == n
        half = [m[: len(m) // 2] for m in msgs]
        h.update(*pack(half))  # host update across both devices
        for k, (i0, i1) in enumerate(((a0, a1), (b0, b1))):
            with torch.cuda.device(k):
                data, off = pack([m[len(m) // 2:] for m in msgs[i0:i1]])
                off = off - off[0]
                td = torch.from_numpy(data).cuda(k)
                to = torch.from_numpy(off.astype(np.int64)).cuda(k)
                h.update_dev(td, to, dev_index=k)
                torch.cuda.synchronize(k)
        got = h.final(512)
        h.close()
        assert np.array_equal(got, orc.kmac_xof_batch(*pack(keys), *pack(msgs), 512, TAG, 512))
    finally:
        e2.close()


# ---- 9. the C++ mirror ---------------------------------------------------------------------------------------------------
def test_cpp_mirror(eng, tmp_path):
    root = os.path.dirname(HERE)
    libdir = os.path.join(root, "capycrypt_b200", "_lib")
    exe = str(tmp_path / "hasher_mirror_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(HERE, "host", "hasher_mirror_check.cpp"),
                    "-L" + libdir, "-lcapycrypt_gpu", "-Wl,-rpath," + os.path.abspath(libdir)], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
