"""GPU: sign and decryption streams fed twice (capy_ed448_sign_stream_new, capy_sponge_decrypt_stream_new,
capy_ed448_key_decrypt_stream_new, capy_hasher_next_pass): messages and ciphertexts fed in pieces, once per pass, give
what the one-shot calls and the oracle give for the concatenated pieces, and a pass 2 over other bytes is caught."""
from __future__ import annotations

import ctypes as C
import importlib.util
import os

import numpy as np
import pytest

from capycrypt_b200 import _binding as B
from capycrypt_b200.api import Gpu, Message, SecParam, Signature
from capycrypt_b200.engine import Engine, pack
from oracle import ref_ed448 as E

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _load(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_S = _load("test_streams_gpu")  # the input generators, and the guarded-buffer and launch-trace helpers
Guarded, _Ptr, _kernels = _S.Guarded, _S._Ptr, _S._kernels
SQ, lengths, plan, oracle_sponge, CUSTOMS = _S.SQ, _S.lengths, _S.plan, _S.oracle_sponge, _S.CUSTOMS


def oracle_open(orc, ct, pw, z, tag, d, variant):
    """sha3/encryptable.rs:58-83 (and the KEM symmetric half) with the C oracle's KMACXOF: (ok, buffer)"""
    ke_c, ka_c = CUSTOMS[variant]
    keymat = orc.kmac_xof(z + pw, b"", 1024, b"S", d)
    pt = bytes(a ^ b for a, b in zip(ct, orc.kmac_xof(keymat[:64], b"", 8 * len(ct), ke_c, d)))
    ok = orc.kmac_xof(keymat[64:], pt, 512, ka_c, d) == tag
    return ok, pt if ok else ct


@pytest.fixture(scope="module")
def eng(engine):
    return engine


@pytest.fixture(scope="module")
def orc(oracle):
    return oracle


def feed(update, ups):
    """every update of a pass; returns the concatenated outputs of update (None: it returns nothing)"""
    n = len(ups[0])
    acc = [bytearray() for _ in range(n)]
    for pieces in ups:
        data, off = pack(pieces)
        r = update(data, off)
        if r is not None:
            for i in range(n):
                acc[i] += r[int(off[i]):int(off[i + 1])].tobytes()
    return [bytes(a) for a in acc]


def sign_stream(eng, pws, msgs, d, rnd, updates=(4, 5), second=None):
    """(h, z, ok) of sign streams; pass 2 feeds `second` (default: msgs) with another chunking"""
    st = eng.ed448_sign_stream(*pack(pws), d)
    with st:
        feed(st.update, plan(rnd, msgs, SQ[d], updates[0]))
        st.next_pass()
        feed(st.update, plan(rnd, msgs if second is None else second, SQ[d], updates[1]))
        return st.final()


def sealed(eng, pws, msgs, nonces, d, variant=B.AE_SHA3):
    md, mo = pack(msgs)
    ct, tag = eng.sponge_encrypt(*pack(pws), nonces, 512, md, mo, d, variant)
    return [ct[int(mo[i]):int(mo[i + 1])].tobytes() for i in range(len(msgs))], tag


def open_stream(st, cts, d, rnd, updates=(4, 5), second=None, in_place=False):
    """(verdicts, pass-2 output, final ok) of a decryption stream"""
    with st:
        feed(st.update, plan(rnd, cts, SQ[d], updates[0]))
        rc1, verdict = st.next_pass()
        if in_place:
            out = feed(lambda data, off: st.decrypt(data, off, out=data), plan(rnd, second or cts, SQ[d], updates[1]))
        else:
            out = feed(st.decrypt, plan(rnd, second or cts, SQ[d], updates[1]))
        rc2, ok = st.final()
        return rc1, verdict.copy(), out, rc2, ok.copy()


# ---- 1. parity ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_sign_parity(eng, d, n):
    rnd = np.random.default_rng(d + n)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [rnd.bytes(int(rnd.integers(0, 20))) for _ in range(n)]
    h, z, ok = sign_stream(eng, pws, msgs, d, rnd)
    wh, wz = eng.ed448_sign(*pack(pws), *pack(msgs), d)
    assert ok.all() and np.array_equal(h, wh) and np.array_equal(z, wz)
    i = n - 1  # the oracle (pure Python Ed448: one item)
    assert (h[i].tobytes(), z[i].tobytes()) == E.sign(pws[i], msgs[i], d)


@pytest.mark.parametrize("variant", [B.AE_SHA3, B.AE_KEM])
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_sponge_decrypt_parity(eng, orc, d, n, variant):
    rnd = np.random.default_rng(3 * d + n + variant)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [rnd.bytes(8) for _ in range(n)]
    nonces = rnd.bytes(512 * n)
    cts, tag = sealed(eng, pws, msgs, nonces, d, variant)
    tag = tag.copy()
    bad = set(range(1, n, 3))  # every third item from the second on: a tampered tag
    for i in bad:
        tag[i, i % 64] ^= 1
    st = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d, variant)
    rc1, verdict, out, rc2, ok = open_stream(st, cts, d, rnd)
    cd, co = pack(cts)
    want, wok = eng.sponge_decrypt(*pack(pws), nonces, 512, cd, co, tag, d, variant)
    assert rc1 == 0 and rc2 == 0
    assert np.array_equal(verdict, wok) and np.array_equal(ok, wok)
    assert b"".join(out) == want.tobytes()
    for i in range(n):
        assert out[i] == (cts[i] if i in bad else msgs[i]), i
    for i in sorted({0, min(1, n - 1), n // 2, n - 1}):  # item 1 (when there is one) has a tampered tag
        zi = nonces[512 * i:512 * (i + 1)]
        assert oracle_sponge(orc, msgs[i], pws[i], zi, d, variant)[0] == cts[i]
        assert oracle_open(orc, cts[i], pws[i], zi, tag[i].tobytes(), d, variant) == (bool(ok[i]), out[i]), i


def key_material(eng, d, n, rnd):
    pws = [b"kd %d" % (i % 7) for i in range(n)]
    pubs = eng.ed448_keygen(*pack(pws), d)
    return pws, pubs, rnd.bytes(56 * n)


@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_key_decrypt_parity(eng, d, n):
    rnd = np.random.default_rng(5 * d + n)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws, pubs, k = key_material(eng, d, n, rnd)
    md, mo = pack(msgs)
    rc, ct, tag, z = eng.ed448_key_encrypt(pubs.tobytes(), k, md, mo, d)
    assert rc == 0
    cts = [ct[int(mo[i]):int(mo[i + 1])].tobytes() for i in range(n)]
    tag = tag.copy()
    for i in range(2, n, 5):
        tag[i, 0] ^= 0x80
    st = eng.ed448_key_decrypt_stream(*pack(pws), z, tag, d)
    rc1, verdict, out, rc2, ok = open_stream(st, cts, d, rnd)
    wrc, want, wok = eng.ed448_key_decrypt(*pack(pws), z, *pack(cts), tag, d)
    assert rc1 == rc2 == wrc == 0
    assert np.array_equal(verdict, wok) and np.array_equal(ok, wok) and b"".join(out) == want.tobytes()
    assert all(out[i] == msgs[i] for i in range(n) if wok[i])
    for i in sorted({0, min(2, n - 1)}):  # the oracle (pure Python Ed448); item 2 has a tampered tag
        Z = E.point_from_bytes(z[i].tobytes())
        assert E.key_decrypt(pws[i], cts[i], d, Z, tag[i].tobytes()) == (bool(ok[i]), out[i]), i


# ---- 2. chunking -------------------------------------------------------------------------------------------------------
def test_kat_sizes_one_byte_per_update(eng):
    """the reference KAT sizes, one byte per update in pass 1, one piece in pass 2 (and the other way round)"""
    rnd = np.random.default_rng(30)
    d = 512
    msgs = [rnd.bytes(L) for L in (0, 1, 135, 136, 137, 200, 272, 273)]
    n = len(msgs)
    L = max(len(m) for m in msgs)
    bytewise = [[m[k:k + 1] for m in msgs] for k in range(L)]
    whole = [msgs]
    pws = [b"kat"] * n
    for first, second in ((bytewise, whole), (whole, bytewise)):
        with eng.ed448_sign_stream(*pack(pws), d) as st:
            feed(st.update, first)
            st.next_pass()
            feed(st.update, second)
            h, z, ok = st.final()
        wh, wz = eng.ed448_sign(*pack(pws), *pack(msgs), d)
        assert ok.all() and np.array_equal(h, wh) and np.array_equal(z, wz)
        nonces = rnd.bytes(512 * n)
        cts, tag = sealed(eng, pws, msgs, nonces, d)
        with eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d) as st:
            feed(st.update, [[c[k:k + 1] for c in cts] for k in range(L)] if first is bytewise else [cts])
            _, verdict = st.next_pass()
            out = feed(st.decrypt, [[c[k:k + 1] for c in cts] for k in range(L)] if second is bytewise else [cts])
            _, ok = st.final()
        assert verdict.all() and ok.all() and out == msgs


# ---- 3. round trips through the Python API -----------------------------------------------------------------------------
def test_round_trips(eng):
    gpu = Gpu(eng)
    rnd = np.random.default_rng(31)
    n, d = 40, SecParam.D384
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[384])]
    ups = plan(rnd, msgs, SQ[384], 4)
    pws = [b"rt %d" % i for i in range(n)]

    with gpu.sha3_encrypt_stream(pws, d) as es:
        cts = [b"".join(p) for p in zip(*[es.update(u) for u in ups])]
        tags = es.finish()
        nonces = es.nonces
    with gpu.sha3_decrypt_stream(pws, nonces, tags, d) as ds:
        for u in plan(rnd, cts, SQ[384], 3):
            ds.update(u)
        assert ds.next_pass() == [None] * n
        pts = [b"".join(p) for p in zip(*[ds.decrypt(u) for u in plan(rnd, cts, SQ[384], 5)])]
        assert ds.finish() == [None] * n and pts == msgs

    kps = gpu.new_keypairs(pws, "rt", d)
    with gpu.key_encrypt_stream([k.pub_key for k in kps], d) as es:
        cts = [b"".join(p) for p in zip(*[es.update(u) for u in ups])]
        tags = es.finish()
        zs = es.asym_nonces
    with gpu.key_decrypt_stream(pws, zs, tags, d) as ds:
        ds.update(cts)
        assert ds.next_pass() == [None] * n
        assert ds.decrypt(cts) == msgs and ds.finish() == [None] * n

    with gpu.sign_stream(kps, d) as ss:
        for u in ups:
            ss.update(u)
        ss.next_pass()
        ss.update(msgs)
        sigs = ss.finish()
    assert all(isinstance(s, Signature) for s in sigs)
    ms = [Message.new(m) for m in msgs]
    for m, s in zip(ms, sigs):
        m.sig, m.d = s, d
    assert gpu.verify(ms, [k.pub_key for k in kps]) == [None] * n
    with gpu.verify_stream(sigs, [k.pub_key for k in kps], d) as vs:
        for u in ups:
            vs.update(u)
        assert vs.finish() == [None] * n
    with pytest.raises(ValueError):
        gpu.sign_stream(kps, SecParam.D224)
    with pytest.raises(ValueError):
        gpu.sha3_decrypt_stream(pws, nonces, tags, SecParam.D224)


# ---- 4. failures -------------------------------------------------------------------------------------------------------
def test_pass_two_differs(eng):
    rnd = np.random.default_rng(32)
    n, d = 8, 256
    msgs = [rnd.bytes(300) for _ in range(n)]
    pws = [rnd.bytes(8) for _ in range(n)]
    flip = bytearray(msgs[1])
    flip[150] ^= 4
    second = list(msgs)
    second[1] = bytes(flip)           # same length, one flipped byte
    second[3] = msgs[3][:-1]          # shorter
    second[5] = msgs[5] + b"\0"       # longer
    changed = {1, 3, 5}

    h, z, ok = sign_stream(eng, pws, msgs, d, rnd, second=second)
    wh, wz = eng.ed448_sign(*pack(pws), *pack(msgs), d)
    for i in range(n):
        if i in changed:
            assert ok[i] == 0 and not h[i].any() and not z[i].any(), i
        else:
            assert ok[i] == 1 and np.array_equal(h[i], wh[i]) and np.array_equal(z[i], wz[i]), i

    nonces = rnd.bytes(512 * n)
    cts, tag = sealed(eng, pws, msgs, nonces, d)
    sc = list(cts)
    for i in changed:
        sc[i] = second[i] if i != 1 else bytes(a ^ b ^ c for a, b, c in zip(cts[1], msgs[1], second[1]))
    sc[3], sc[5] = cts[3][:-1], cts[5] + b"\0"
    st = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
    rc1, verdict, out, rc2, ok = open_stream(st, cts, d, rnd, second=sc)
    assert verdict.all()
    assert [int(o) for o in ok] == [0 if i in changed else 1 for i in range(n)]
    assert out[0] == msgs[0]


def test_tampered_ciphertext_and_off_curve(eng):
    rnd = np.random.default_rng(33)
    n, d = 6, 512
    msgs = [rnd.bytes(200) for _ in range(n)]
    pws = [b"t"] * n
    nonces = rnd.bytes(512 * n)
    cts, tag = sealed(eng, pws, msgs, nonces, d)
    cts[2] = cts[2][:10] + bytes([cts[2][10] ^ 1]) + cts[2][11:]
    st = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
    _, verdict, out, _, ok = open_stream(st, cts, d, rnd, in_place=True)
    assert list(verdict) == [1, 1, 0, 1, 1, 1] and list(ok) == list(verdict)
    assert out[2] == cts[2] and out[0] == msgs[0]

    kp, pubs, k = key_material(eng, d, n, rnd)
    md, mo = pack(msgs)
    _, ct, ktag, z = eng.ed448_key_encrypt(pubs.tobytes(), k, md, mo, d)
    z = z.copy()
    z[4, 0] ^= 1  # off the curve
    st = eng.ed448_key_decrypt_stream(*pack(kp), z, ktag, d)
    kcts = [ct[int(mo[i]):int(mo[i + 1])].tobytes() for i in range(n)]
    rc1, verdict, out, rc2, ok = open_stream(st, kcts, d, rnd)
    assert rc1 == B.ERR_BAD_POINT and rc2 == B.ERR_BAD_POINT
    assert verdict[4] == 0 and ok[4] == 0 and out[4] == kcts[4]
    assert all(verdict[i] and ok[i] and out[i] == msgs[i] for i in range(n) if i != 4)


# ---- 5. buffers ----------------------------------------------------------------------------------------------------------
def test_in_place(eng):
    rnd = np.random.default_rng(34)
    n, d = 257, 256
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [b"x"] * n
    nonces = rnd.bytes(512 * n)
    cts, tag = sealed(eng, pws, msgs, nonces, d)
    st = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
    _, verdict, out, _, ok = open_stream(st, cts, d, rnd, in_place=True)
    assert verdict.all() and ok.all() and out == msgs


@pytest.mark.parametrize("offset", [0, 1, 3])
def test_dev_guarded(eng, offset):
    import torch

    rnd = np.random.default_rng(35 + offset)
    n, d = 129, 512
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [rnd.bytes(5) for _ in range(n)]
    nonces = rnd.bytes(512 * n)
    cts, tag = sealed(eng, pws, msgs, nonces, d)
    tag = tag.copy()
    tag[7, 3] ^= 1
    st = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
    for j, pieces in enumerate(plan(rnd, cts, SQ[d], 4)):
        data, off = pack(pieces)
        gd = Guarded(len(data), offset, data, seed=j)
        go = Guarded(8 * (n + 1), 8 * offset, off.tobytes(), seed=100 + j)
        st.update_dev(_Ptr(gd.ptr), _Ptr(go.ptr))
        torch.cuda.synchronize()
        assert np.array_equal(gd.get(), data)
        go.get()
    gv = Guarded(n, offset, seed=5)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    st.next_pass_dev(_Ptr(gv.ptr), flag)
    torch.cuda.synchronize()
    verdict = gv.get()
    out = [bytearray() for _ in range(n)]
    for j, pieces in enumerate(plan(rnd, cts, SQ[d], 5)):
        data, off = pack(pieces)
        gd = Guarded(len(data), offset, data, seed=10 + j)
        go = Guarded(8 * (n + 1), 8 * offset, off.tobytes(), seed=110 + j)
        gc = Guarded(len(data), offset + 2, seed=210 + j)
        st.decrypt_dev(_Ptr(gd.ptr), _Ptr(go.ptr), _Ptr(gc.ptr))
        torch.cuda.synchronize()
        go.get()
        c = gc.get()
        for i in range(n):
            out[i] += c[int(off[i]):int(off[i + 1])].tobytes()
    gok = Guarded(n, offset, seed=6)
    st.final_dev(_Ptr(gok.ptr), flag)
    torch.cuda.synchronize()
    ok = gok.get()
    st.close()
    assert int(flag.item()) == 0
    assert [int(v) for v in verdict] == [0 if i == 7 else 1 for i in range(n)] and np.array_equal(ok, verdict)
    assert all(bytes(out[i]) == (cts[i] if i == 7 else msgs[i]) for i in range(n))

    sw = eng.ed448_sign_stream(*pack(pws), d)
    for p in range(2):
        for j, pieces in enumerate(plan(rnd, msgs, SQ[d], 3)):
            data, off = pack(pieces)
            gd = Guarded(len(data), offset, data, seed=300 + j)
            go = Guarded(8 * (n + 1), 8 * offset, off.tobytes(), seed=400 + j)
            sw.update_dev(_Ptr(gd.ptr), _Ptr(go.ptr))
            torch.cuda.synchronize()
            go.get()
        if p == 0:
            sw.next_pass_dev()
    gh, gz, gk = Guarded(56 * n, offset, seed=1), Guarded(56 * n, offset + 1, seed=2), Guarded(n, offset, seed=3)
    sw.final_dev(_Ptr(gh.ptr), _Ptr(gz.ptr), _Ptr(gk.ptr))
    torch.cuda.synchronize()
    sw.close()
    wh, wz = eng.ed448_sign(*pack(pws), *pack(msgs), d)
    assert gk.get().all() and np.array_equal(gh.get().reshape(n, 56), wh) and np.array_equal(gz.get().reshape(n, 56), wz)


# ---- 6. launches ---------------------------------------------------------------------------------------------------------
def test_launches(eng, tmp_path):
    rnd = np.random.default_rng(36)
    n = 300
    msgs = [rnd.bytes(int(x)) for x in rnd.integers(0, 700, size=n)]
    data, off = pack(msgs)
    pws = [b"p"] * n
    for d, L in ((256, 21), (384, 19), (512, 17)):
        nonces = rnd.bytes(512 * n)
        cts, tag = sealed(eng, pws, msgs, nonces, d)
        cd, co = pack(cts)
        st = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
        assert _kernels(lambda: st.update(cd, co), tmp_path) == [f"sponge_chain_kernel<{L}>"]
        ks = _kernels(lambda: st.next_pass(), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>", "ae_finish_kernel"], ks
        assert _kernels(lambda: st.decrypt(cd, co), tmp_path) == [f"sponge_chain_kernel<{L}>"]
        ks = _kernels(lambda: st.final(), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>", "ae_finish_kernel"], ks
        st.close()
        sw = eng.ed448_sign_stream(*pack(pws), d)
        assert _kernels(lambda: sw.update(data, off), tmp_path) == [f"sponge_chain_kernel<{L}>"]
        ks = _kernels(lambda: sw.next_pass(), tmp_path)
        assert ks[0] == f"sponge_chain_kernel<{L}>" and ks[-2:] == [f"sponge_chain_kernel<{L}>"] * 2, ks
        assert _kernels(lambda: sw.update(data, off), tmp_path) == [f"sponge_chain_kernel<{L}>"]
        ks = _kernels(lambda: sw.final(), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>"] * 2 + ["verify_compare_kernel", "sign_finish_kernel"], ks
        sw.close()


# ---- 7. isolation from the one-shot calls --------------------------------------------------------------------------------
def test_isolation(eng):
    rnd = np.random.default_rng(37)
    n, d = 1000, 512
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [rnd.bytes(8) for _ in range(n)]
    nonces = rnd.bytes(512 * n)
    cts, tag = sealed(eng, pws, msgs, nonces, d)
    other = [rnd.bytes(int(x)) for x in rnd.integers(0, 5000, size=n)]
    od, oo = pack(other)

    def noise():
        eng.sponge_encrypt(*pack(pws), nonces, 512, od, oo, d)
        eng.ed448_sign(*pack(pws), od, oo, d)
        eng.kmac_xof(*pack(pws), od, oo, 448, b"N", d)

    ds = eng.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
    sw = eng.ed448_sign_stream(*pack(pws), d)
    for pieces_c, pieces_m in zip(plan(rnd, cts, SQ[d], 3), plan(rnd, msgs, SQ[d], 3)):
        ds.update(*pack(pieces_c))
        sw.update(*pack(pieces_m))
        noise()
    _, verdict = ds.next_pass()
    sw.next_pass()
    noise()
    out = [bytearray() for _ in range(n)]
    for pieces_c, pieces_m in zip(plan(rnd, cts, SQ[d], 4), plan(rnd, msgs, SQ[d], 4)):
        data, off = pack(pieces_c)
        r = ds.decrypt(data, off)
        for i in range(n):
            out[i] += r[int(off[i]):int(off[i + 1])].tobytes()
        sw.update(*pack(pieces_m))
        noise()
    _, ok = ds.final()
    h, z, sok = sw.final()
    ds.close()
    sw.close()
    wh, wz = eng.ed448_sign(*pack(pws), *pack(msgs), d)
    assert verdict.all() and ok.all() and [bytes(o) for o in out] == msgs
    assert sok.all() and np.array_equal(h, wh) and np.array_equal(z, wz)


# ---- 8. errors ---------------------------------------------------------------------------------------------------------------
def test_errors(eng):
    lib, ctx = eng.lib, eng._ctx
    n, d = 3, 256
    pws = [b"a", b"b", b"c"]
    pd, po = pack(pws)
    nonces = bytes(512 * n)
    tags = bytes(64 * n)
    hp = C.c_void_p()
    u8 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint8))  # noqa: E731
    u64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint64))  # noqa: E731
    tb = np.frombuffer(tags, np.uint8).copy()
    zb = np.frombuffer(nonces, np.uint8).copy()
    # creation
    assert lib.capy_ed448_sign_stream_new(ctx, 224, u8(pd), u64(po), n, C.byref(hp)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_sign_stream_new(ctx, 100, u8(pd), u64(po), n, C.byref(hp)) == B.ERR_BAD_SECPARAM
    assert lib.capy_sponge_decrypt_stream_new(ctx, 224, B.AE_SHA3, u8(pd), u64(po), u8(zb), 512, u8(tb), n,
                                              C.byref(hp)) == B.ERR_BAD_ARG
    assert lib.capy_sponge_decrypt_stream_new(ctx, d, 7, u8(pd), u64(po), u8(zb), 512, u8(tb), n,
                                              C.byref(hp)) == B.ERR_BAD_ARG
    assert lib.capy_sponge_decrypt_stream_new(ctx, 100, B.AE_SHA3, u8(pd), u64(po), u8(zb), 512, u8(tb), n,
                                              C.byref(hp)) == B.ERR_BAD_SECPARAM
    z112 = np.zeros(112 * n, np.uint8)
    assert lib.capy_ed448_key_decrypt_stream_new(ctx, 224, u8(pd), u64(po), u8(z112), u8(tb), n,
                                                 C.byref(hp)) == B.ERR_BAD_ARG
    data, off = pack([b"xy", b"", b"z"])
    out = np.zeros_like(data)
    ok = np.zeros(n, np.uint8)
    h56, z56 = np.zeros(56 * n, np.uint8), np.zeros(56 * n, np.uint8)

    ds = eng.sponge_decrypt_stream(pd, po, nonces, 512, tags, d)
    sw = eng.ed448_sign_stream(pd, po, d)
    old = eng.sha3_hasher(n, d)
    es = eng.sponge_encrypt_stream(pd, po, nonces, 512, d)
    H = lambda s: s.handle  # noqa: E731
    # pass 1: decrypt_update, finals, the other kinds' calls
    assert lib.capy_hasher_decrypt_update(ctx, H(ds), u8(data), u64(off), u8(out)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_final(ctx, H(ds), u8(ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_sign_final(ctx, H(sw), u8(h56), u8(z56), u8(ok)) == B.ERR_BAD_ARG
    for s in (ds, sw):
        assert lib.capy_hasher_final(ctx, H(s), 448, None, u8(h56)) == B.ERR_BAD_ARG
        assert lib.capy_hasher_final(ctx, H(s), 512, None, u8(h56)) == B.ERR_BAD_ARG
        assert lib.capy_hasher_verify_final(ctx, H(s), u8(ok)) == B.ERR_BAD_ARG
        assert lib.capy_hasher_encrypt_update(ctx, H(s), u8(data), u64(off), u8(out)) == B.ERR_BAD_ARG
    for s in (old, es):
        assert lib.capy_hasher_next_pass(ctx, H(s), None) == B.ERR_BAD_ARG
        assert lib.capy_hasher_decrypt_update(ctx, H(s), u8(data), u64(off), u8(out)) == B.ERR_BAD_ARG
        assert lib.capy_hasher_decrypt_final(ctx, H(s), u8(ok)) == B.ERR_BAD_ARG
        assert lib.capy_hasher_sign_final(ctx, H(s), u8(h56), u8(z56), u8(ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_sign_final(ctx, H(ds), u8(h56), u8(z56), u8(ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_final(ctx, H(sw), u8(ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_next_pass(ctx, H(sw), u8(ok)) == B.ERR_BAD_ARG  # sign: ok must be NULL
    # another ctx
    e2 = Engine()
    try:
        assert lib.capy_hasher_next_pass(e2._ctx, H(ds), None) == B.ERR_BAD_ARG
    finally:
        e2.close()
    # pass 2
    ds.update(data, off)
    sw.update(data, off)
    assert lib.capy_hasher_next_pass(ctx, H(ds), None) == 0
    assert lib.capy_hasher_next_pass(ctx, H(sw), None) == 0
    assert lib.capy_hasher_next_pass(ctx, H(ds), None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_next_pass(ctx, H(sw), None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_update(ctx, H(ds), u8(data), u64(off)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_update(ctx, H(sw), u8(data), u64(off)) == 0
    assert lib.capy_hasher_decrypt_update(ctx, H(ds), u8(data), u64(off), u8(out)) == 0
    assert lib.capy_hasher_decrypt_final(ctx, H(ds), u8(ok)) == 0
    assert lib.capy_hasher_sign_final(ctx, H(sw), u8(h56), u8(z56), u8(ok)) == 0
    # after the final
    assert lib.capy_hasher_decrypt_update(ctx, H(ds), u8(data), u64(off), u8(out)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_final(ctx, H(ds), u8(ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_update(ctx, H(sw), u8(data), u64(off)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_sign_final(ctx, H(sw), u8(h56), u8(z56), u8(ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_next_pass(ctx, H(sw), None) == B.ERR_BAD_ARG
    for s in (ds, sw, old, es):
        s.close()

    # the _dev forms keep the pass of their device
    import torch

    st = torch.cuda.current_stream().cuda_stream
    t_data = torch.from_numpy(data).cuda()
    t_off = torch.from_numpy(off.astype(np.int64)).cuda()
    t_out = torch.empty_like(t_data)
    t_ok, t_h, t_z = (torch.zeros(n * w, dtype=torch.uint8, device="cuda") for w in (1, 56, 56))
    P = lambda t: t.data_ptr()  # noqa: E731
    ds = eng.sponge_decrypt_stream(pd, po, nonces, 512, tags, d)
    sw = eng.ed448_sign_stream(pd, po, d)
    es = eng.sponge_encrypt_stream(pd, po, nonces, 512, d)
    assert lib.capy_hasher_decrypt_update_dev(ctx, H(ds), 0, st, P(t_data), P(t_off), P(t_out)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_final_dev(ctx, H(ds), 0, st, P(t_ok), None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_sign_final_dev(ctx, H(sw), 0, st, P(t_h), P(t_z), P(t_ok)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_next_pass_dev(ctx, H(sw), 0, st, P(t_ok), None) == B.ERR_BAD_ARG  # sign: no ok
    assert lib.capy_hasher_next_pass_dev(ctx, H(es), 0, st, None, None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_next_pass_dev(ctx, H(ds), 1 << 20, st, None, None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_update_dev(ctx, H(ds), 0, st, P(t_data), P(t_off)) == 0
    assert lib.capy_hasher_next_pass_dev(ctx, H(ds), 0, st, P(t_ok), None) == 0
    assert lib.capy_hasher_next_pass_dev(ctx, H(sw), 0, st, None, None) == 0
    assert lib.capy_hasher_next_pass_dev(ctx, H(ds), 0, st, P(t_ok), None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_next_pass_dev(ctx, H(sw), 0, st, None, None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_update_dev(ctx, H(ds), 0, st, P(t_data), P(t_off)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_update_dev(ctx, H(sw), 0, st, P(t_data), P(t_off), P(t_out)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_update_dev(ctx, H(ds), 0, st, P(t_data), P(t_off), P(t_out)) == 0
    assert lib.capy_hasher_decrypt_final_dev(ctx, H(ds), 0, st, P(t_ok), None) == 0
    assert lib.capy_hasher_sign_final_dev(ctx, H(sw), 0, st, P(t_h), P(t_z), P(t_ok)) == 0
    assert lib.capy_hasher_decrypt_update_dev(ctx, H(ds), 0, st, P(t_data), P(t_off), P(t_out)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_decrypt_final_dev(ctx, H(ds), 0, st, P(t_ok), None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_update_dev(ctx, H(sw), 0, st, P(t_data), P(t_off)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_sign_final_dev(ctx, H(sw), 0, st, P(t_h), P(t_z), P(t_ok)) == B.ERR_BAD_ARG
    torch.cuda.synchronize()
    for s in (ds, sw, es):
        s.close()
    # n = 0 works end to end
    with eng.ed448_sign_stream(*pack([]), d) as s0:
        s0.next_pass()
        h, z, ok0 = s0.final()
        assert h.shape == (0, 56)


# ---- 9. scale ----------------------------------------------------------------------------------------------------------------
def test_scale_2e16_streams(eng, orc):
    """2^16 decryption and sign streams x 16 updates of 4 KiB per pass through the _dev calls, against the one-shot
    calls on the 64 KiB messages"""
    import torch

    n, d, piece, ups = 1 << 16, 512, 4096, 16
    g = torch.Generator(device="cuda").manual_seed(38)
    msgs = torch.randint(0, 256, (n, ups * piece), dtype=torch.uint8, device="cuda", generator=g)
    pws = [b"scale %d" % i for i in range(n)]
    nonces = np.random.default_rng(38).bytes(512 * n)
    pd, po = pack(pws)
    t_pd, t_po = torch.from_numpy(pd).cuda(), torch.from_numpy(po.astype(np.int64)).cuda()
    t_nonce = torch.from_numpy(np.frombuffer(nonces, np.uint8).copy()).cuda()
    flat = msgs.reshape(-1)
    moff = torch.arange(n + 1, dtype=torch.int64, device="cuda") * (ups * piece)
    ct = torch.empty_like(flat)
    tag = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    eng.sponge_encrypt_dev(t_pd, t_po, len(pd), t_nonce, 512, flat, moff, d, ct, tag)
    tag[5, 0] ^= 1
    want = torch.empty_like(flat)
    wok = torch.empty(n, dtype=torch.uint8, device="cuda")
    eng.sponge_decrypt_dev(t_pd, t_po, len(pd), t_nonce, 512, ct, moff, tag, d, want, wok)
    ct2 = ct.reshape(n, -1)
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * piece
    out = torch.empty_like(ct2)
    verdict = torch.empty(n, dtype=torch.uint8, device="cuda")
    ok = torch.empty(n, dtype=torch.uint8, device="cuda")
    with eng.sponge_decrypt_stream(pd, po, nonces, 512, tag.cpu().numpy(), d) as st:
        for k in range(ups):
            st.update_dev(ct2[:, k * piece:(k + 1) * piece].contiguous(), off)
        st.next_pass_dev(verdict)
        for k in range(ups):
            src = ct2[:, k * piece:(k + 1) * piece].contiguous()
            st.decrypt_dev(src, off, src)
            out[:, k * piece:(k + 1) * piece] = src
        st.final_dev(ok)
        torch.cuda.synchronize()
    assert torch.equal(verdict, wok) and torch.equal(ok, wok) and int(wok.sum()) == n - 1
    assert torch.equal(out.reshape(-1), want)
    assert torch.equal(out[0], msgs[0]) and torch.equal(out[5], ct2[5])

    h = torch.empty((n, 56), dtype=torch.uint8, device="cuda")
    z, sok = torch.empty_like(h), torch.empty(n, dtype=torch.uint8, device="cuda")
    with eng.ed448_sign_stream(pd, po, d) as sw:
        for p in range(2):
            for k in range(ups):
                sw.update_dev(msgs[:, k * piece:(k + 1) * piece].contiguous(), off)
            if p == 0:
                sw.next_pass_dev()
        sw.final_dev(h, z, sok)
        torch.cuda.synchronize()
    wh, wz = torch.empty_like(h), torch.empty_like(h)
    eng.ed448_sign_dev(t_pd, t_po, flat, moff, d, wh, wz)
    torch.cuda.synchronize()
    assert bool(sok.all()) and torch.equal(h, wh) and torch.equal(z, wz)


# ---- 10. two devices -----------------------------------------------------------------------------------------------------------
def test_two_devices():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    e2 = Engine([0, 1])
    try:
        rnd = np.random.default_rng(39)
        n, d = 301, 512
        msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
        pws = [rnd.bytes(9) for _ in range(n)]
        nonces = rnd.bytes(512 * n)
        cts, tag = sealed(e2, pws, msgs, nonces, d)
        st = e2.sponge_decrypt_stream(*pack(pws), nonces, 512, tag, d)
        (a0, a1), (b0, b1) = st.device_range(0), st.device_range(1)
        assert a0 == 0 and a1 == b0 and b1 == n
        _, verdict, out, _, ok = open_stream(st, cts, d, rnd)
        assert verdict.all() and ok.all() and out == msgs
        h, z, sok = sign_stream(e2, pws, msgs, d, rnd)
        wh, wz = e2.ed448_sign(*pack(pws), *pack(msgs), d)
        assert sok.all() and np.array_equal(h, wh) and np.array_equal(z, wz)
    finally:
        e2.close()


# ---- 11. the C++ mirror -----------------------------------------------------------------------------------------------------------
def test_cpp_mirror(eng, tmp_path):
    import subprocess

    root = os.path.dirname(HERE)
    libdir = os.path.join(root, "capycrypt_b200", "_lib")
    exe = str(tmp_path / "two_pass_mirror_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(HERE, "host", "two_pass_mirror_check.cpp"),
                    "-L" + libdir, "-lcapycrypt_gpu", "-Wl,-rpath," + os.path.abspath(libdir)], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
