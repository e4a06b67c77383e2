"""GPU: prepared public keys (capy_ed448_pub_prepare and the *_prepared entry points).

Every prepared call must give byte for byte what the per-item-key call gives with the key repeated n times -- and the
oracle -- for every on-curve key: keys of order r run the comb path (one joint fixed_base_kernel launch for verify, two
for key_encrypt, no var_base_kernel), a key with a torsion component the variable-base fallback."""
import ctypes as C
import importlib.util
import json
import os
import subprocess

import numpy as np
import pytest

from capycrypt_b200 import _binding as B
from capycrypt_b200.engine import pack
from oracle import ref_ed448 as E

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
R = E.R
GUARD = 4096


def _matrix():
    spec = importlib.util.spec_from_file_location("dispatch_matrix", os.path.join(HERE, "test_dispatch_matrix_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture(scope="module")
def signers(engine):
    """d -> (password, public key, prepared key): the key pair depends on the security parameter"""
    made = {}

    def get(d):
        if d not in made:
            pw = b"release signing key"
            pub = engine.ed448_keygen(*pack([pw]), d)[0].tobytes()
            made[d] = (pw, pub, engine.ed448_pub_prepare(pub))
        return made[d]

    yield get
    for _, _, key in made.values():
        key.close()


@pytest.fixture(scope="module")
def signer(signers):
    return signers(512)


def _batch(engine, pw, d, n, seed):
    """n signatures by pw over 1..300-byte messages, with h, z or the message altered on some items, h + r (unreduced,
    quirk Q10) and z + r (>= r) on others"""
    rnd = np.random.default_rng(seed)
    lens = rnd.integers(1, 300, size=n)
    msgs, moff = pack([rnd.integers(0, 256, size=int(k), dtype=np.uint8).tobytes() for k in lens])
    h, z = engine.ed448_sign(*pack([pw] * n), msgs, moff, d)
    h, z, msgs = h.copy(), z.copy(), msgs.copy()
    for i in range(n):
        kind = (i + seed) % 7 if n > 1 else 0
        if kind == 1:
            h[i, 3] ^= 0x40
        elif kind == 2:
            z[i, 55] ^= 1
        elif kind == 3:
            msgs[int(moff[i])] ^= 0x80
        elif kind in (4, 5):
            row = h if kind == 4 else z
            v = int.from_bytes(row[i].tobytes(), "big") + R
            if v < 2**448:
                row[i] = np.frombuffer(v.to_bytes(56, "big"), np.uint8)
    return msgs, moff, h, z


@pytest.mark.parametrize("d", [224, 256, 384, 512])
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
def test_verify_prepared_equals_verify_and_oracle(engine, oracle, signers, d, n):
    pw, pub, key = signers(d)
    msgs, moff, h, z = _batch(engine, pw, d, n, seed=d + n)
    pubs = np.frombuffer(pub * n, np.uint8)
    ok = engine.ed448_verify_prepared(key, msgs, moff, h, z, d)
    rc, want = engine.ed448_verify(pubs, msgs, moff, h, z, d)
    assert rc == 0
    assert np.array_equal(ok, want), np.nonzero(ok != want)[0][:10]
    assert np.array_equal(ok, oracle.verify_batch(pubs, msgs, moff, h, z, d, threads=0))
    if n > 1:
        assert ok.any() and not ok.all()


@pytest.mark.parametrize("d", [224, 512])
def test_key_encrypt_prepared_equals_key_encrypt_and_decrypts(engine, signers, d):
    pw, pub, key = signers(d)
    n = 129
    rnd = np.random.default_rng(d)
    msgs, moff = pack([rnd.integers(0, 256, size=int(k), dtype=np.uint8).tobytes() for k in rnd.integers(0, 600, size=n)])
    k = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
    ct, tag, zp = engine.ed448_key_encrypt_prepared(key, k, msgs, moff, d)
    rc, ct0, tag0, z0 = engine.ed448_key_encrypt(pub * n, k, msgs, moff, d)
    assert rc == 0
    assert np.array_equal(ct, ct0) and np.array_equal(tag, tag0) and np.array_equal(zp, z0)
    for i in (0, 5, n - 1):
        m = msgs[int(moff[i]):int(moff[i + 1])].tobytes()
        c_ref, t_ref, z_ref = E.key_encrypt(E.point_from_bytes(pub), m, d, k[56 * i:56 * i + 56].tobytes())
        assert ct[int(moff[i]):int(moff[i + 1])].tobytes() == c_ref and tag[i].tobytes() == t_ref
        assert zp[i].tobytes() == E.point_to_bytes(z_ref)
    _, out, ok = engine.ed448_key_decrypt(*pack([pw] * n), zp, ct, moff, tag, d)
    assert ok.all() and np.array_equal(out, msgs)


def _special_keys():
    s = 0x1234567890ABCDEF
    torsion = E.point_add(E.scalar_mult(s, E.GENERATOR), (1, 0))  # (1, 0) has order 4
    return {"G": (E.GENERATOR, 1), "identity": (E.IDENTITY, 1), "torsion": (torsion, 0)}


@pytest.mark.parametrize("which", ["G", "identity", "torsion", "keygen"])
def test_special_keys_same_bytes(engine, oracle, signer, which):
    if which == "keygen":
        pub, comb = signer[1], 1
    else:
        pt, comb = _special_keys()[which]
        pub = E.point_to_bytes(pt)
    d, n = 256, 300
    rnd = np.random.default_rng(7)
    msgs, moff = pack([rnd.integers(0, 256, size=int(k), dtype=np.uint8).tobytes() for k in rnd.integers(0, 200, size=n)])
    h = rnd.integers(0, 256, size=(n, 56), dtype=np.uint8)
    z = rnd.integers(0, 256, size=(n, 56), dtype=np.uint8)
    k = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
    if which == "G":  # some valid signatures against G: the secret scalar is 1 (z = k - h mod r with U = [k]G)
        for i in range(0, n, 3):
            kk = int.from_bytes(k[56 * i:56 * i + 56].tobytes(), "big") % R
            ux = E.point_to_bytes(E.scalar_mult(kk, E.GENERATOR))[:56]
            hh = oracle.kmac_xof(ux, msgs[int(moff[i]):int(moff[i + 1])].tobytes(), 448, b"T", d)
            h[i] = np.frombuffer(hh, np.uint8)
            z[i] = np.frombuffer(((kk - int.from_bytes(hh, "big")) % R).to_bytes(56, "big"), np.uint8)
    pubs = np.frombuffer(pub * n, np.uint8)
    with engine.ed448_pub_prepare(pub) as key:
        assert key.uses_comb == bool(comb)
        ok = engine.ed448_verify_prepared(key, msgs, moff, h, z, d)
        rc, want = engine.ed448_verify(pubs, msgs, moff, h, z, d)
        assert rc == 0 and np.array_equal(ok, want)
        assert np.array_equal(ok, oracle.verify_batch(pubs, msgs, moff, h, z, d, threads=0))
        if which == "G":
            assert ok[::3].all()
        ct, tag, zp = engine.ed448_key_encrypt_prepared(key, k, msgs, moff, d)
        rc, ct0, tag0, z0 = engine.ed448_key_encrypt(pubs, k, msgs, moff, d)
        assert rc == 0
        assert np.array_equal(ct, ct0) and np.array_equal(tag, tag0) and np.array_equal(zp, z0)


def test_off_curve_key_is_refused_without_a_handle(engine, signer):
    b = bytearray(signer[1])
    b[60] ^= 0x10
    assert not E.on_curve(E.point_from_bytes(bytes(b)))
    h = C.c_void_p(12345)
    raw = np.frombuffer(bytes(b), np.uint8)
    assert engine.lib.capy_ed448_pub_prepare(engine._ctx, raw.ctypes.data, C.byref(h)) == B.ERR_BAD_POINT
    assert not h.value
    with pytest.raises(B.CapyError) as e:
        engine.ed448_pub_prepare(bytes(b))
    assert e.value.status == B.ERR_BAD_POINT


def test_key_of_another_ctx_is_bad_arg(engine, signer):
    import torch

    from capycrypt_b200 import Engine

    pw, pub, key = signer
    other = Engine()
    try:
        msgs, moff, h, z = _batch(engine, pw, 256, 3, seed=1)
        ok = np.zeros(3, np.uint8)
        assert other.lib.capy_ed448_verify_prepared_batch(other._ctx, 256, key.handle, msgs.ctypes.data, moff.ctypes.data,
                                                          h.ctypes.data, z.ctypes.data, 3, ok.ctypes.data) == B.ERR_BAD_ARG
        ct, tag, zp = np.zeros(len(msgs), np.uint8), np.zeros(3 * 56, np.uint8), np.zeros(3 * 112, np.uint8)
        kr = np.zeros(3 * 56, np.uint8)
        assert other.lib.capy_ed448_key_encrypt_prepared_batch(other._ctx, 256, key.handle, kr.ctypes.data, msgs.ctypes.data,
                                                               moff.ctypes.data, 3, ct.ctypes.data, tag.ctypes.data,
                                                               zp.ctypes.data) == B.ERR_BAD_ARG
        dm, dh, dz = (torch.from_numpy(a.reshape(-1).copy()).cuda() for a in (msgs, h, z))
        doff = torch.from_numpy(moff.astype(np.int64)).cuda()
        dok = torch.zeros(3, dtype=torch.uint8, device="cuda")
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        assert other.lib.capy_ed448_verify_prepared_batch_dev(other._ctx, 0, stream, 256, key.handle, dm.data_ptr(),
                                                              doff.data_ptr(), dh.data_ptr(), dz.data_ptr(), 3,
                                                              dok.data_ptr()) == B.ERR_BAD_ARG
    finally:
        other.close()


# ---- _dev twins: inputs and outputs cut out of guarded device buffers ------------------------------------------------
class Guarded:
    """`nbytes` of device memory at `offset` inside a buffer with GUARD bytes of a seeded pattern on each side"""

    def __init__(self, nbytes, offset, fill=None, seed=0):
        import torch

        self.lo, self.hi = GUARD + offset, GUARD + offset + nbytes
        host = np.random.default_rng(seed * 131 + offset).integers(0, 256, size=self.hi + GUARD, dtype=np.uint8)
        if fill is not None:
            host[self.lo:self.hi] = np.asarray(fill, dtype=np.uint8).reshape(-1)
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


def _stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _launched(tmp_path, fn):
    """capy:: kernels fn launched, in order (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    m = _matrix()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    path = tmp_path / f"trace{len(list(tmp_path.iterdir()))}.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    ks = [m.normalise_kernel(e["name"]) for e in events if e.get("cat") == "kernel" and "capy::" in e.get("name", "")]
    assert ks and set(ks) <= m.KERNELS, ks
    return ks


@pytest.mark.parametrize("offset", [0, 1])
def test_dev_twins_guarded_and_launch_path(engine, signer, tmp_path, offset):
    import torch

    pw, pub, key = signer
    d, n = 512, 257
    msgs, moff, h, z = _batch(engine, pw, d, n, seed=offset)
    pubs = np.frombuffer(pub * n, np.uint8)
    rc, want_ok = engine.ed448_verify(pubs, msgs, moff, h, z, d)
    m_g, h_g, z_g = Guarded(len(msgs), offset, msgs, 1), Guarded(h.size, offset, h, 2), Guarded(z.size, offset, z, 3)
    ok_g = Guarded(n, offset, seed=4)
    moff_t = torch.from_numpy(moff.astype(np.int64)).cuda()
    ks = _launched(tmp_path, lambda: engine._check(engine.lib.capy_ed448_verify_prepared_batch_dev(
        engine._ctx, 0, _stream(), d, key.handle, m_g.ptr, moff_t.data_ptr(), h_g.ptr, z_g.ptr, n, ok_g.ptr)))
    assert ks.count("fixed_base_kernel") == 1 and "var_base_kernel" not in ks, ks
    assert np.array_equal(ok_g.get(), want_ok)
    for g in (m_g, h_g, z_g):
        g.get()

    k = np.random.default_rng(offset).integers(0, 256, size=n * 56, dtype=np.uint8)
    _, ct0, tag0, zp0 = engine.ed448_key_encrypt(pubs, k, msgs, moff, d)
    k_g = Guarded(k.size, offset, k, 5)
    ct_g, tag_g, zp_g = Guarded(len(msgs), offset, seed=6), Guarded(n * 56, offset, seed=7), Guarded(n * 112, offset, seed=8)
    ks = _launched(tmp_path, lambda: engine._check(engine.lib.capy_ed448_key_encrypt_prepared_batch_dev(
        engine._ctx, 0, _stream(), d, key.handle, k_g.ptr, m_g.ptr, moff_t.data_ptr(), n, ct_g.ptr, tag_g.ptr, zp_g.ptr)))
    assert ks.count("fixed_base_kernel") == 2 and "var_base_kernel" not in ks, ks
    assert np.array_equal(ct_g.get(), ct0)
    assert np.array_equal(tag_g.get(), tag0.reshape(-1)) and np.array_equal(zp_g.get(), zp0.reshape(-1))
    k_g.get()


def test_dev_twins_fallback_key(engine, tmp_path):
    """a key with a torsion component: the _dev twins broadcast it and run the variable-base pipelines"""
    import torch

    pub = E.point_to_bytes(_special_keys()["torsion"][0])
    d, n = 256, 77
    rnd = np.random.default_rng(9)
    msgs, moff = pack([rnd.integers(0, 256, size=int(k), dtype=np.uint8).tobytes() for k in rnd.integers(0, 90, size=n)])
    h = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
    z = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
    pubs = np.frombuffer(pub * n, np.uint8)
    _, want_ok = engine.ed448_verify(pubs, msgs, moff, h, z, d)
    with engine.ed448_pub_prepare(pub) as key:
        assert not key.uses_comb
        m_g, h_g, z_g, ok_g = Guarded(len(msgs), 3, msgs), Guarded(h.size, 3, h), Guarded(z.size, 3, z), Guarded(n, 3)
        moff_t = torch.from_numpy(moff.astype(np.int64)).cuda()
        ks = _launched(tmp_path, lambda: engine._check(engine.lib.capy_ed448_verify_prepared_batch_dev(
            engine._ctx, 0, _stream(), d, key.handle, m_g.ptr, moff_t.data_ptr(), h_g.ptr, z_g.ptr, n, ok_g.ptr)))
        assert "var_base_kernel" in ks, ks
        assert np.array_equal(ok_g.get(), want_ok)


def test_large_batch_against_oracle_sample(engine, oracle, signer):
    pw, pub, key = signer
    d, n = 512, 1 << 18
    rnd = np.random.default_rng(18)
    msgs = rnd.integers(0, 256, size=n * 256, dtype=np.uint8)
    moff = np.arange(n + 1, dtype=np.uint64) * 256
    h, z = engine.ed448_sign(*pack([pw] * n), msgs, moff, d)
    h, z = h.copy(), z.copy()
    h[1::3, 0] ^= 1
    ok = engine.ed448_verify_prepared(key, msgs, moff, h, z, d)
    idx = np.array(sorted(set(rnd.choice(n, size=300, replace=False).tolist()) | {0, n - 1}))
    sm, so = pack([msgs[int(moff[i]):int(moff[i + 1])] for i in idx])
    want = oracle.verify_batch(np.frombuffer(pub * len(idx), np.uint8), sm, so, h[idx], z[idx], d, threads=0)
    assert np.array_equal(ok[idx], want)
    assert ok[0::3].all() and not ok[1::3].any()


def test_two_device_ctx_same_bytes(engine, signer):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from capycrypt_b200 import Engine

    pw, pub, key = signer
    d, n = 256, 5000
    msgs, moff, h, z = _batch(engine, pw, d, n, seed=2)
    want = engine.ed448_verify_prepared(key, msgs, moff, h, z, d)
    k = np.random.default_rng(2).integers(0, 256, size=n * 56, dtype=np.uint8)
    want_e = engine.ed448_key_encrypt_prepared(key, k, msgs, moff, d)
    two = Engine([0, 1])
    try:
        with two.ed448_pub_prepare(pub) as key2:
            assert np.array_equal(two.ed448_verify_prepared(key2, msgs, moff, h, z, d), want)
            for a, b in zip(two.ed448_key_encrypt_prepared(key2, k, msgs, moff, d), want_e):
                assert np.array_equal(a, b)
    finally:
        two.close()


def test_python_api_one_signer_one_recipient(engine, signer):
    from capycrypt_b200.api import Gpu, Message, OperationError

    pw, pub, _ = signer
    gpu = Gpu(engine)
    msgs = [Message.new(bytes([i]) * (10 + i)) for i in range(6)]
    kp = gpu.new_keypairs([pw], "signer", 512)[0]
    gpu.sign(msgs, [kp] * len(msgs), 512)
    msgs[2].msg[0] ^= 1
    msgs[4].sig = None
    with gpu.prepare_public_key(pub) as key:
        got = gpu.verify_prepared(msgs, key)
        want = gpu.verify(msgs, [pub] * len(msgs))
        assert [type(e).__name__ + (e.kind if e else "") for e in got] == \
            [type(e).__name__ + (e.kind if e else "") for e in want]
        assert got[0] is None and got[2].kind == "SignatureVerificationFailure" and got[4].kind == "SignatureNotSet"
        a = [Message.new(b"x" * (50 * i)) for i in range(4)]
        b = [Message.new(b"x" * (50 * i)) for i in range(4)]
        ks = [bytes([7 + i]) * 56 for i in range(4)]
        gpu.key_encrypt_prepared(a, key, 512, k_rand=ks)
        gpu.key_encrypt(b, [pub] * 4, 512, k_rand=ks)
        assert [(m.msg, m.digest, m.asym_nonce) for m in a] == [(m.msg, m.digest, m.asym_nonce) for m in b]
        assert gpu.key_decrypt(a, [pw] * 4) == [None] * 4
    bad = bytearray(pub)
    bad[60] ^= 0x10
    with pytest.raises(OperationError):
        gpu.prepare_public_key(bytes(bad))


def test_cpp_mirror_prepared_key(tmp_path):
    root = os.path.join(HERE, "..")
    libdir = os.path.abspath(os.path.join(root, "capycrypt_b200", "_lib"))
    exe = str(tmp_path / "prepared_mirror_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(HERE, "host", "prepared_mirror_check.cpp"),
                    "-L" + libdir, "-lcapycrypt_gpu", "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "prepared mirror ok" in r.stdout, r.stdout + r.stderr
