"""GPU: checkpoints and forks of SHA3-d and KMACXOF streams (capy_hasher_export / _import / _fork).  A stream exported
and imported (into another engine), or forked, continues as the original would: its final is, byte for byte, the one-shot
call and the oracle on everything fed before and after."""
from __future__ import annotations

import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

from capycrypt_b200 import _binding as B
from capycrypt_b200.api import Gpu, SecParam
from capycrypt_b200.engine import Engine, hasher_blob_info, pack

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
SHA3_RATE = {224: 144, 256: 136, 384: 104, 512: 72}
KMAC_RATE = {256: 168, 384: 152, 512: 136}
Q3_KEYS = {256: (163, 331), 384: (147, 299), 512: (131, 267)}  # key lengths whose bytepad content is a multiple of w
TAG = b"My Tagged Application"
KINDS = [("sha3", d) for d in SHA3_RATE] + [("kmac", d) for d in KMAC_RATE]
OUT_BITS = 1000  # KMACXOF output length of these tests: not a multiple of the rate


@pytest.fixture(scope="module")
def eng():
    import torch

    assert torch.cuda.is_available(), "-m gpu tests need a CUDA device"
    torch.cuda.set_device(0)
    e = Engine()
    yield e
    e.close()


@pytest.fixture(scope="module")
def orc():
    from oracle import cpu

    return cpu.get()


# ---- inputs ---------------------------------------------------------------------------------------------------------
def rate_of(kind, d):
    return SHA3_RATE[d] if kind == "sha3" else KMAC_RATE[d]


def lengths(rnd, n, r):
    """message lengths with the edge cases up front: empty, r - 1, r, r + 1, len % 136 == 135, 2 r - 1, 2 r"""
    edge = [0, r - 1, r, r + 1, 135, 271, 2 * r - 1, 2 * r, 1, 3 * r + 5]
    return [edge[i] if i < len(edge) else int(rnd.integers(0, 3 * r + 8)) for i in range(n)]


def cut_points(rnd, msgs, r):
    """where each message is checkpointed: edge offsets (0, r - 1, r, r + 1, the end) up front, then seeded"""
    pts = []
    for i, m in enumerate(msgs):
        edge = [0, r - 1, r, r + 1, len(m)]
        p = edge[i % len(edge)] if i < 3 * len(edge) else int(rnd.integers(0, len(m) + 1))
        pts.append(min(p, len(m)))
    return pts


def chunking(rnd, length, r, updates):
    """`updates` piece lengths that add up to `length`, cuts at 1, r - 1, r, r + 1 when they fit, empty pieces seeded"""
    cuts = {c for c in (1, r - 1, r, r + 1) if 0 < c < length}
    while len(cuts) < updates - 2 and len(cuts) < length - 1:
        cuts.add(int(rnd.integers(1, length)))
    cuts = sorted(cuts)[: updates - 1]
    bounds = [0] + cuts + [length]
    lens = [b - a for a, b in zip(bounds, bounds[1:])]
    while len(lens) < updates:
        lens.insert(int(rnd.integers(0, len(lens) + 1)), 0)
    return lens


def feed(h, parts, rnd, r, updates):
    """feeds parts[i] to stream i in `updates` calls"""
    plan = [chunking(rnd, len(p), r, updates) for p in parts]
    pos = [0] * len(parts)
    for k in range(updates):
        pieces = []
        for i, p in enumerate(parts):
            pieces.append(p[pos[i]:pos[i] + plan[i][k]])
            pos[i] += plan[i][k]
        h.update(*pack(pieces))


def kmac_keys(rnd, n, d):
    q = Q3_KEYS[d]
    edge = [b"", bytes(q[0]), bytes(range(256))[: q[1]], bytes(q[1])]
    return [edge[i] if i < len(edge) else rnd.bytes(int(rnd.integers(0, 80))) for i in range(n)]


class Case:
    """one kind and d: how to make its hasher, finish it, and what the one-shot call and the oracle give"""

    def __init__(self, kind, d, n, rnd):
        self.kind, self.d, self.n, self.r = kind, d, n, rate_of(kind, d)
        self.keys = kmac_keys(rnd, n, d) if kind == "kmac" else None

    def make(self, e, keys=None):
        if self.kind == "sha3":
            return e.sha3_hasher(self.n if keys is None else len(keys), self.d)
        return e.kmac_xof_hasher(*pack(self.keys if keys is None else keys), TAG, self.d)

    def final(self, h):
        return h.final() if self.kind == "sha3" else h.final(OUT_BITS)

    def want(self, e, orc, msgs, keys=None):
        """(one-shot, oracle) for msgs; keys: the key of every message (default: the case's own)"""
        data, off = pack(msgs)
        if self.kind == "sha3":
            return e.sha3(data, off, self.d), orc.sha3_batch(data, off, self.d, threads=orc.max_threads)
        kd, ko = pack(self.keys if keys is None else keys)
        return (e.kmac_xof(kd, ko, data, off, OUT_BITS, TAG, self.d),
                orc.kmac_xof_batch(kd, ko, data, off, OUT_BITS, TAG, self.d, threads=orc.max_threads))

    def check(self, got, e, orc, msgs, keys=None):
        one, ref = self.want(e, orc, msgs, keys)
        assert np.array_equal(got, one)
        assert np.array_equal(got, ref)


def records(blob, r):
    """(lanes, totals, carries) of a blob's records"""
    rec = 208 + r
    n = (len(blob) - 64) // rec
    a = np.frombuffer(bytes(blob), np.uint8)[64:].reshape(n, rec)
    return a[:, :200], a[:, 200:208].copy().view("<u8").reshape(-1), a[:, 208:]


# ---- 1. round trip through a blob into a new engine --------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("kind,d", KINDS)
def test_round_trip(orc, kind, d, n):
    rnd = np.random.default_rng(d * 13 + n + (kind == "kmac"))
    cs = Case(kind, d, n, rnd)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, cs.r)]
    pts = cut_points(rnd, msgs, cs.r)
    e1 = Engine()
    h = cs.make(e1)
    feed(h, [m[:p] for m, p in zip(msgs, pts)], rnd, cs.r, 4)
    blob = h.export()
    h.close()
    e1.close()
    assert blob.size == 64 + n * (208 + cs.r)
    assert hasher_blob_info(blob) == (int(kind == "kmac"), d, n)
    _, totals, carries = records(blob, cs.r)
    assert totals.tolist() == pts
    for i in range(min(n, 64)):
        assert not carries[i, pts[i] % cs.r:].any(), "the carry tail is exported as zero"
    e2 = Engine()
    try:
        h2 = e2.import_hasher(blob)
        assert (h2.n, h2.d, h2.kmac) == (n, d, kind == "kmac")
        feed(h2, [m[p:] for m, p in zip(msgs, pts)], rnd, cs.r, 3)
        got = cs.final(h2)
        h2.close()
        cs.check(got, e2, orc, msgs)
    finally:
        e2.close()


# ---- 2. canonical blobs ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,d", [("sha3", 256), ("sha3", 224), ("kmac", 512), ("kmac", 256)])
def test_canonical_blobs(eng, kind, d):
    rnd = np.random.default_rng(d + 5)
    n = 300
    cs = Case(kind, d, n, rnd)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, cs.r)]
    blobs = []
    for updates in (1, 3, 7):  # whole, and cut two different ways
        with cs.make(eng) as h:
            feed(h, msgs, rnd, cs.r, updates)
            blobs.append(h.export())
    assert np.array_equal(blobs[0], blobs[1]) and np.array_equal(blobs[0], blobs[2])
    with eng.import_hasher(blobs[1]) as h:
        assert np.array_equal(h.export(), blobs[1]), "export -> import -> export is the identity"


# ---- 3. forks ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,d", [("sha3", 256), ("sha3", 512), ("kmac", 256), ("kmac", 384)])
def test_fork_maps(eng, orc, kind, d):
    rnd = np.random.default_rng(d * 3 + (kind == "kmac"))
    n = 129
    cs = Case(kind, d, n, rnd)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, cs.r)]
    pts = cut_points(rnd, msgs, cs.r)
    pre = [m[:p] for m, p in zip(msgs, pts)]
    maps = {
        "identity": list(range(n)),
        "reverse": list(range(n))[::-1],
        "replicate one": [5] * 300,
        "seeded repeats": rnd.integers(0, n, size=200).tolist(),
        "empty": [],
    }
    with cs.make(eng) as h:
        feed(h, pre, rnd, cs.r, 3)
        kids = {name: h.fork(src) for name, src in maps.items()}
        # every child and the parent continue with suffixes of their own
        for name, src in maps.items():
            k = kids[name]
            assert k.n == len(src) and k.d == d
            suf = [rnd.bytes(int(rnd.integers(0, 2 * cs.r + 3))) for _ in src]
            feed(k, suf, rnd, cs.r, 3)
            got = cs.final(k)
            k.close()
            if not src:
                assert got.shape[0] == 0
                continue
            keys = [cs.keys[s] for s in src] if cs.keys else None
            cs.check(got, eng, orc, [pre[s] + x for s, x in zip(src, suf)], keys)
        feed(h, [m[p:] for m, p in zip(msgs, pts)], rnd, cs.r, 2)
        cs.check(cs.final(h), eng, orc, msgs)  # the parent is unaffected by its children


def test_siblings_and_parent_independent(eng, orc):
    rnd = np.random.default_rng(77)
    n, d = 64, 256
    cs = Case("sha3", d, n, rnd)
    pre = [rnd.bytes(int(rnd.integers(0, 400))) for _ in range(n)]
    src = list(range(n))
    with cs.make(eng) as h:
        h.update(*pack(pre))
        a, b = h.fork(src), h.fork(src)
        sa = [rnd.bytes(100) for _ in range(n)]
        sb = [rnd.bytes(37) for _ in range(n)]
        a.update(*pack(sa))
        b.update(*pack(sb))
        c = a.fork(src[::-1])  # a fork of a fork
        sp = [rnd.bytes(300) for _ in range(n)]
        h.update(*pack(sp))
        cs.check(a.final(), eng, orc, [p + x for p, x in zip(pre, sa)])
        cs.check(b.final(), eng, orc, [p + x for p, x in zip(pre, sb)])
        cs.check(c.final(), eng, orc, [pre[j] + sa[j] for j in src[::-1]])
        cs.check(h.final(), eng, orc, [p + x for p, x in zip(pre, sp)])
        for k in (a, b, c):
            k.close()


def test_copy_finish_is_the_digest_so_far(eng, orc):
    """api: s.copy().finish() mid-stream gives the one-shot digest of the prefix, and s goes on"""
    rnd = np.random.default_rng(9)
    gpu = Gpu(eng)
    n = 200
    msgs = [rnd.bytes(int(L)) for L in rnd.integers(0, 700, size=n)]
    cut = [int(rnd.integers(0, len(m) + 1)) for m in msgs]
    keys = [rnd.bytes(int(rnd.integers(0, 64))) for _ in range(n)]
    with gpu.sha3_stream(n, SecParam.D256) as s, gpu.kmac_xof_stream(keys, TAG, SecParam.D512) as k:
        for st in (s, k):
            st.update([m[:c] for m, c in zip(msgs, cut)])
        with s.copy() as c1, k.copy() as c2:
            mid_s, mid_k = c1.finish(), c2.finish(512)
        pre = pack([m[:c] for m, c in zip(msgs, cut)])
        assert mid_s == [r.tobytes() for r in orc.sha3_batch(*pre, 256)]
        assert mid_k == [r.tobytes() for r in orc.kmac_xof_batch(*pack(keys), *pre, 512, TAG, 512)]
        blob = k.export()
        for st in (s, k):
            st.update([m[c:] for m, c in zip(msgs, cut)])
        assert s.finish() == [r.tobytes() for r in orc.sha3_batch(*pack(msgs), 256)]
        want_k = [r.tobytes() for r in orc.kmac_xof_batch(*pack(keys), *pack(msgs), 512, TAG, 512)]
        assert k.finish(512) == want_k
    with gpu.resume_stream(blob) as r:
        with r.fork([3, 3, 0]) as f:
            f.update([msgs[3][cut[3]:], msgs[3][cut[3]:], msgs[0][cut[0]:]])
            assert f.finish(512) == [want_k[3], want_k[3], want_k[0]]
        r.update([m[c:] for m, c in zip(msgs, cut)])
        assert r.finish(512) == want_k


# ---- 4. isolation from the one-shot calls -------------------------------------------------------------------------------
def test_isolation(eng, orc):
    rnd = np.random.default_rng(17)
    n = 1000
    cs = Case("kmac", 512, n, rnd)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, cs.r)]
    pts = cut_points(rnd, msgs, cs.r)
    big = 1 << 16  # one-shot batches large enough for the chain-cut and dependent-job launches (their scratch slots)
    bd = rnd.integers(0, 256, size=big * 2048, dtype=np.uint8)
    bo = np.arange(big + 1, dtype=np.uint64) * 2048
    bk, bko = pack([b"k" * 32] * big)
    pw, pwo = pack([b"pw"] * big)
    nonces = rnd.integers(0, 256, size=big * 16, dtype=np.uint8)
    mm = rnd.integers(0, 256, size=big * 64, dtype=np.uint8)
    mo = np.arange(big + 1, dtype=np.uint64) * 64

    def noise():
        eng.sha3(bd, bo, 256)
        eng.kmac_xof(bk, bko, bd, bo, 512, TAG, 512)
        ct, tags = eng.sponge_encrypt(pw, pwo, nonces, 16, mm, mo, 512)
        out, ok = eng.sponge_decrypt(pw, pwo, nonces, 16, ct, mo, tags, 512)
        assert ok.all() and np.array_equal(out, mm)

    h = cs.make(eng)
    feed(h, [m[:p] for m, p in zip(msgs, pts)], rnd, cs.r, 2)
    noise()
    blob = h.export()
    noise()
    h2 = eng.import_hasher(blob)
    noise()
    f = h.fork(list(range(n)))
    noise()
    rest = [m[p:] for m, p in zip(msgs, pts)]
    for x in (h, h2, f):
        x.update(*pack(rest))
        noise()
    for x in (h, h2, f):
        cs.check(cs.final(x), eng, orc, msgs)
        x.close()


# ---- 5. several devices --------------------------------------------------------------------------------------------------
def _device_sets():
    import torch

    sets = [[0, 0], [0, 0, 0]]  # a ctx over one GPU twice runs every multi-device path
    if torch.cuda.device_count() >= 2:
        sets.append([0, 1])
    return sets


@pytest.mark.parametrize("devices", _device_sets(), ids=lambda s: "-".join(map(str, s)))
def test_across_devices(orc, devices):
    rnd = np.random.default_rng(len(devices) * 31 + devices[-1])
    n = 301
    cs = Case("kmac", 384, n, rnd)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, cs.r)]
    pts = cut_points(rnd, msgs, cs.r)
    pre, rest = [m[:p] for m, p in zip(msgs, pts)], [m[p:] for m, p in zip(msgs, pts)]
    multi, single = Engine(devices), Engine()
    try:
        h = cs.make(multi)
        assert h.device_range(len(devices) - 1)[1] == n and h.device_range(0)[1] < n
        feed(h, pre, rnd, cs.r, 3)
        blob = h.export()
        with cs.make(single) as s:  # the same streams on one device export the same blob
            feed(s, pre, rnd, cs.r, 2)
            assert np.array_equal(s.export(), blob)
        # multi -> single and single -> multi
        with single.import_hasher(blob) as h1, multi.import_hasher(h.export()) as hm:
            assert np.array_equal(hm.export(), blob)
            for x in (h1, hm):
                x.update(*pack(rest))
                cs.check(cs.final(x), single, orc, msgs)
        # forks whose sources sit on the other devices: reversed, one item replicated, seeded with repeats
        for src in (list(range(n))[::-1], [n - 1] * 250, rnd.integers(0, n, size=400).tolist(), [0]):
            with h.fork(src) as f:
                assert f.device_range(len(devices) - 1)[1] == len(src)
                f.update(*pack([rest[s] for s in src]))
                cs.check(cs.final(f), single, orc, [msgs[s] for s in src], [cs.keys[s] for s in src])
        h.update(*pack(rest))
        cs.check(cs.final(h), single, orc, msgs)
        h.close()
    finally:
        multi.close()
        single.close()


# ---- 6. size ------------------------------------------------------------------------------------------------------------------
def test_scale_2e20_streams(orc):
    n, d, r = 1 << 20, 256, 136
    rnd = np.random.default_rng(2)
    sample = np.array(sorted({0, n - 1} | set(rnd.choice(n, 200, replace=False).tolist())))
    a_len, b_len = 200, 90  # mid-message: 64 carry bytes after the first piece
    first = rnd.integers(0, 256, size=n * a_len, dtype=np.uint8)
    second = rnd.integers(0, 256, size=n * b_len, dtype=np.uint8)
    oa = np.arange(n + 1, dtype=np.uint64) * a_len
    ob = np.arange(n + 1, dtype=np.uint64) * b_len
    src = rnd.integers(0, n, size=n).astype(np.uint64)
    src[:3] = [n - 1, 0, n - 1]

    def msg(i, j):  # stream i's first piece, then the second piece of slot j
        return first[i * a_len:(i + 1) * a_len].tobytes() + second[j * b_len:(j + 1) * b_len].tobytes()

    e1 = Engine()
    h = e1.sha3_hasher(n, d)
    h.update(first, oa)
    blob = h.export()
    h.close()
    e1.close()
    e2 = Engine()
    try:
        h2 = e2.import_hasher(blob)
        f = h2.fork(src)
        for x in (h2, f):
            x.update(second, ob)
        got_h, got_f = h2.final(), f.final()
        h2.close()
        f.close()
    finally:
        e2.close()
    want_h = orc.sha3_batch(*pack([msg(i, i) for i in sample]), d)
    want_f = orc.sha3_batch(*pack([msg(int(src[j]), j) for j in sample]), d)
    assert np.array_equal(got_h[sample], want_h)
    assert np.array_equal(got_f[sample], want_f)


# ---- 7. errors ------------------------------------------------------------------------------------------------------------
def _refused(lib, ctx, h, n):
    """export_size, export and fork of h all return ERR_BAD_ARG, and fork leaves *out NULL"""
    size = C.c_uint64(0)
    assert lib.capy_hasher_export_size(h, C.byref(size)) == B.ERR_BAD_ARG
    buf = np.zeros(64 + max(n, 1) * 400, np.uint8)
    assert lib.capy_hasher_export(ctx, h, buf.ctypes.data, buf.size) == B.ERR_BAD_ARG
    src = np.zeros(max(n, 1), np.uint64)
    out = C.c_void_p(12345)
    assert lib.capy_hasher_fork(ctx, h, src.ctypes.data, src.size, C.byref(out)) == B.ERR_BAD_ARG
    assert not out.value


def test_refused_kinds(eng):
    import torch

    lib, ctx = eng.lib, eng._ctx
    rnd = np.random.default_rng(4)
    n = 3
    pw, pwo = pack([b"pw%d" % i for i in range(n)])
    nonces = rnd.integers(0, 256, size=n * 512, dtype=np.uint8)
    pub = eng.ed448_keygen(pw, pwo, 256)
    streams = {
        "encrypt": eng.sponge_encrypt_stream(pw, pwo, nonces, 512, 256),
        "key_encrypt": eng.ed448_key_encrypt_stream(pub, rnd.bytes(56 * n), 256)[0],
        "verify": eng.ed448_verify_stream(pub, bytes(56 * n), bytes(56 * n), 256),
        "sign": eng.ed448_sign_stream(pw, pwo, 256),
        "decrypt": eng.sponge_decrypt_stream(pw, pwo, nonces, 512, bytes(64 * n), 256),
    }
    for name, st in streams.items():
        _refused(lib, ctx, st.handle, n)
        st.close()
    # finished: by the host final, and by the _dev final of the only device
    with eng.sha3_hasher(n, 256) as h:
        h.final()
        _refused(lib, ctx, h.handle, n)
    with eng.kmac_xof_hasher(*pack([b"k"] * n), b"", 256) as h:
        out = torch.zeros(n, 32, dtype=torch.uint8, device="cuda")
        h.final_dev(out, 256)
        torch.cuda.synchronize()
        _refused(lib, ctx, h.handle, n)


def test_argument_errors(eng):
    lib, ctx = eng.lib, eng._ctx
    n = 5
    out = C.c_void_p(12345)
    with eng.sha3_hasher(n, 384) as h:
        h.update(*pack([b"x" * i for i in range(n)]))
        size = C.c_uint64(0)
        assert lib.capy_hasher_export_size(h.handle, C.byref(size)) == B.OK and size.value == 64 + n * 312
        buf = np.zeros(size.value, np.uint8)
        assert lib.capy_hasher_export(ctx, h.handle, buf.ctypes.data, size.value - 1) == B.ERR_BAD_ARG
        assert lib.capy_hasher_export(ctx, h.handle, None, size.value) == B.ERR_BAD_ARG
        for src in ([n], [0, n + 5], [2**64 - 1]):
            s = np.array(src, np.uint64)
            assert lib.capy_hasher_fork(ctx, h.handle, s.ctypes.data, s.size, C.byref(out)) == B.ERR_BAD_ARG
            assert not out.value
            out = C.c_void_p(12345)
        assert lib.capy_hasher_fork(ctx, h.handle, None, 1, C.byref(out)) == B.ERR_BAD_ARG and not out.value
        assert lib.capy_hasher_fork(ctx, h.handle, None, 0, None) == B.ERR_BAD_ARG
        other = Engine()
        try:  # a hasher of another ctx
            assert lib.capy_hasher_export(other._ctx, h.handle, buf.ctypes.data, buf.size) == B.ERR_BAD_ARG
            s = np.zeros(1, np.uint64)
            out = C.c_void_p(12345)
            assert lib.capy_hasher_fork(other._ctx, h.handle, s.ctypes.data, 1, C.byref(out)) == B.ERR_BAD_ARG
            assert not out.value
        finally:
            other.close()
        h.update(*pack([b"y"] * n))  # still usable after the refusals
        assert np.array_equal(h.final(), eng.sha3(*pack([b"x" * i + b"y" for i in range(n)]), 384))
    with eng.sha3_hasher(0, 256) as h0:
        s = np.zeros(1, np.uint64)
        out = C.c_void_p(12345)
        assert lib.capy_hasher_fork(ctx, h0.handle, s.ctypes.data, 1, C.byref(out)) == B.ERR_BAD_ARG and not out.value
        with h0.fork([]) as f0:
            assert f0.n == 0 and f0.final().shape == (0, 32)
        blob = h0.export()
        assert blob.size == 64
        with eng.import_hasher(blob) as i0:
            assert i0.n == 0


def _import_rc(eng, blob: bytes):
    a = np.frombuffer(blob, np.uint8) if blob else np.zeros(1, np.uint8)
    out = C.c_void_p(12345)
    rc = eng.lib.capy_hasher_import(eng._ctx, a.ctypes.data, len(blob), C.byref(out))
    if rc == B.OK:
        eng.lib.capy_hasher_free(out)
    else:
        assert not out.value
    return rc


def test_malformed_blobs(eng):
    rnd = np.random.default_rng(6)
    n = 4
    with eng.kmac_xof_hasher(*pack([b"key"] * n), TAG, 512) as h:
        h.update(*pack([rnd.bytes(L) for L in (0, 10, 136, 140)]))  # carries of 0, 10, 0 and 4 bytes
        good = h.export().tobytes()
    assert _import_rc(eng, good) == B.OK
    rec = 208 + 136

    def patch(b, at, fmt, v):
        b = bytearray(b)
        struct.pack_into(fmt, b, at, v)
        return bytes(b)

    bad = {
        "magic": b"capyhstr" + good[8:],
        "version": patch(good, 8, "<I", 2),
        "kind": patch(good, 12, "<I", 7),
        "d": patch(good, 16, "<I", 300),
        "kmac d224": patch(patch(patch(good, 16, "<I", 224), 20, "<I", 172), 24, "<I", 380),
        "kind of another rate": patch(good, 12, "<I", 0),
        "rate": patch(good, 20, "<I", 144),
        "record": patch(good, 24, "<I", rec + 8),
        "zero field": patch(good, 28, "<I", 1),
        "reserved": patch(good, 63, "<B", 1),
        "n": patch(good, 32, "<Q", n + 1),
        "short": good[:-1],
        "long": good + b"\0",
        "header only": good[:64],
        "empty": b"",
        # carry tails: item 1 holds 10 carry bytes, item 0 none, item 3 four
        "tail after 10": patch(good, 64 + rec + 208 + 10, "<B", 1),
        "tail of an empty carry": patch(good, 64 + 208, "<B", 0x80),
        "last tail byte": patch(good, 64 + 4 * rec - 1, "<B", 1),
        "tail after 4": patch(good, 64 + 3 * rec + 208 + 4, "<B", 1),
    }
    for name, b in bad.items():
        assert _import_rc(eng, b) == B.ERR_BAD_ARG, name
    # the bytes inside the carry and anything in the lanes and totals are the caller's business
    assert _import_rc(eng, patch(good, 64 + rec + 208 + 9, "<B", 0xFF)) == B.OK
    assert _import_rc(eng, patch(good, 64 + 7, "<B", 0xFF)) == B.OK


# ---- 8. the C++ mirror -----------------------------------------------------------------------------------------------------
def test_cpp_mirror(eng, tmp_path):
    root = os.path.dirname(HERE)
    libdir = os.path.join(root, "capycrypt_b200", "_lib")
    exe = str(tmp_path / "hasher_checkpoint_mirror_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(HERE, "host", "hasher_checkpoint_mirror_check.cpp"),
                    "-L" + libdir, "-lcapycrypt_gpu", "-Wl,-rpath," + os.path.abspath(libdir)], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
