"""GPU: encryption and verification streams (capy_sponge_encrypt_stream_new, capy_ed448_key_encrypt_stream_new,
capy_ed448_verify_stream_new): plaintexts and messages fed in pieces give, byte for byte, what the one-shot calls and
the oracle give for the concatenated pieces."""
from __future__ import annotations

import ctypes as C
import functools
import importlib.util
import json
import os
import subprocess

import numpy as np
import pytest

from capycrypt_b200 import _binding as B
from capycrypt_b200.engine import Engine, pack
from oracle import ref_ed448 as E
from oracle import ref_sha3

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _hasher_tests():
    """the guarded-buffer and launch-trace helpers of test_hasher_gpu.py"""
    spec = importlib.util.spec_from_file_location("hasher_tests", os.path.join(HERE, "test_hasher_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_H = _hasher_tests()
Guarded, _Ptr, _kernels = _H.Guarded, _H._Ptr, _H._kernels


@functools.lru_cache(maxsize=None)
def _torsion():
    """the signing helpers of test_ed448_torsion_gpu.py (loaded when first used: that module loads this one)"""
    spec = importlib.util.spec_from_file_location("torsion_tests", os.path.join(HERE, "test_ed448_torsion_gpu.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


TORSION_S = 0x1234567890ABCDEF  # the secret scalar of the torsion key [s]G + (1, 0)
SQ = {256: 168, 384: 152, 512: 136}  # squeeze width of the keystream = rate of the tag and "T" streams
CUSTOMS = {B.AE_SHA3: (b"SKE", b"SKA"), B.AE_KEM: (b"KEMKE", b"KEMKA")}


@pytest.fixture(scope="module")
def eng(engine):
    return engine


@pytest.fixture(scope="module")
def orc(oracle):
    return oracle


@pytest.fixture(scope="module")
def keys(eng):
    """d -> (passwords, their public keys, a prepared key with a comb table (of pws[0]), a prepared torsion key)"""
    made = {}
    torsion = E.point_to_bytes(E.point_add(E.scalar_mult(TORSION_S, E.GENERATOR), (1, 0)))  # (1, 0) has order 4

    def get(d):
        if d not in made:
            pws = [b"stream key %d" % i for i in range(64)]
            pubs = eng.ed448_keygen(*pack(pws), d)
            comb = eng.ed448_pub_prepare(pubs[0].tobytes())
            tors = eng.ed448_pub_prepare(torsion)
            assert comb.uses_comb and not tors.uses_comb
            made[d] = (pws, pubs, comb, tors)
        return made[d]

    yield get
    for _, _, a, b in made.values():
        a.close()
        b.close()


# ---- inputs ------------------------------------------------------------------------------------------------------------
def lengths(rnd, n, r):
    """plaintext lengths with the edge cases up front: empty, around one and two blocks, odd"""
    edge = [0, 1, r - 1, r, r + 1, 2 * r - 1, 2 * r, 2 * r + 1, 7, 3 * r + 5]
    return [edge[i] if i < len(edge) else int(rnd.integers(0, 3 * r + 8)) for i in range(n)]


def chunking(rnd, length, r, updates):
    """`updates` piece lengths that add up to `length`.  Cuts on a block boundary and one byte either side of it (the
    squeeze block and the tag rate have the same width), odd cuts (keystream positions with pos % 8 != 0), the rest
    seeded; the remaining pieces are empty, at seeded places"""
    cuts = {c for c in (1, 3, r - 1, r, r + 1, 2 * r - 1, 2 * r, 2 * r + 1) if 0 < c < length}
    while len(cuts) < updates - 2 and len(cuts) < length - 1:
        cuts.add(int(rnd.integers(1, length)))
    cuts = sorted(cuts)[: updates - 1]
    bounds = [0] + cuts + [length]
    lens = [b - a for a, b in zip(bounds, bounds[1:])]
    while len(lens) < updates:
        lens.insert(int(rnd.integers(0, len(lens) + 1)), 0)
    return lens


def plan(rnd, msgs, r, updates):
    """the pieces of every update: [update][item] -> bytes"""
    cuts = [chunking(rnd, len(m), r, updates) for m in msgs]
    pos = [0] * len(msgs)
    out = []
    for k in range(updates):
        pieces = []
        for i, m in enumerate(msgs):
            pieces.append(m[pos[i]:pos[i] + cuts[i][k]])
            pos[i] += cuts[i][k]
        out.append(pieces)
    return out


def seal(st, pieces_per_update):
    """feeds every update through an EncryptStream; returns the concatenated ciphertext of every item and the tags"""
    n = len(pieces_per_update[0])
    ct = [bytearray() for _ in range(n)]
    for pieces in pieces_per_update:
        data, off = pack(pieces)
        c = st.update(data, off)
        for i in range(n):
            ct[i] += c[int(off[i]):int(off[i + 1])].tobytes()
    return [bytes(c) for c in ct], st.final()


def oracle_sponge(orc, msg, pw, z, d, variant):
    """sha3/encryptable.rs:29-45 (and the KEM symmetric half) with the C oracle's KMACXOF"""
    ke_c, ka_c = CUSTOMS[variant]
    keymat = orc.kmac_xof(z + pw, b"", 1024, b"S", d)
    ks = orc.kmac_xof(keymat[:64], b"", 8 * len(msg), ke_c, d)
    return bytes(a ^ b for a, b in zip(msg, ks)), orc.kmac_xof(keymat[64:], msg, 512, ka_c, d)


# ---- 1. parity: sponge AE ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [B.AE_SHA3, B.AE_KEM])
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_sponge_parity(eng, orc, d, n, variant):
    rnd = np.random.default_rng(d * 13 + n + variant)
    r = SQ[d]
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, r)]
    pws = [rnd.bytes(int(rnd.integers(0, 40))) for _ in range(n)]
    nonces = rnd.bytes(512 * n)
    pd, po = pack(pws)
    with eng.sponge_encrypt_stream(pd, po, nonces, 512, d, variant) as st:
        ct, tag = seal(st, plan(rnd, msgs, r, 7))
    md, mo = pack(msgs)
    want_ct, want_tag = eng.sponge_encrypt(pd, po, nonces, 512, md, mo, d, variant)
    assert b"".join(ct) == want_ct.tobytes()
    assert np.array_equal(tag, want_tag)
    for i in sorted({0, n // 2, n - 1}):
        z = nonces[512 * i:512 * (i + 1)]
        assert (ct[i], tag[i].tobytes()) == oracle_sponge(orc, msgs[i], pws[i], z, d, variant), i
        if variant == B.AE_SHA3 and len(msgs[i]) < 400:
            assert (ct[i], tag[i].tobytes()) == ref_sha3.sha3_encrypt(msgs[i], pws[i], d, z), i


# ---- 2. parity: key_encrypt ----------------------------------------------------------------------------------------------
def key_form(keys, d, form, n):
    """(argument of the stream calls, n x 112 key bytes the one-shot per-item call takes)"""
    pws, pubs, comb, tors = keys(d)
    if form == "pub":
        pub = np.concatenate([pubs[i % len(pubs)] for i in range(n)]).reshape(n, 112)
        return pub, pub
    key = comb if form == "comb" else tors
    return key, np.tile(np.frombuffer(key.pub_xy112, np.uint8), (n, 1))


@pytest.mark.parametrize("form", ["pub", "comb", "torsion"])
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_key_encrypt_parity(eng, keys, d, n, form):
    rnd = np.random.default_rng(d * 17 + n)
    r = SQ[d]
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, r)]
    k = rnd.bytes(56 * n)
    arg, pub = key_form(keys, d, form, n)
    st, z = eng.ed448_key_encrypt_stream(arg, k, d)
    with st:
        ct, tag = seal(st, plan(rnd, msgs, r, 6))
    md, mo = pack(msgs)
    rc, want_ct, want_tag, want_z = eng.ed448_key_encrypt(pub.reshape(-1), k, md, mo, d)
    assert rc == 0
    assert b"".join(ct) == want_ct.tobytes() and np.array_equal(tag, want_tag) and np.array_equal(z, want_z)
    if form != "pub":
        p_ct, p_tag, p_z = eng.ed448_key_encrypt_prepared(arg, k, md, mo, d)
        assert b"".join(ct) == p_ct.tobytes() and np.array_equal(tag, p_tag) and np.array_equal(z, p_z)
    i = n - 1  # the oracle (pure Python Ed448: one item)
    oc, ot, oz = E.key_encrypt(E.point_from_bytes(pub[i].tobytes()), msgs[i], d, k[56 * i:56 * (i + 1)])
    assert (ct[i], tag[i].tobytes(), z[i].tobytes()) == (oc, ot, E.point_to_bytes(oz))


# ---- 3. parity: verify ---------------------------------------------------------------------------------------------------
def signed(eng, orc, keys, d, n, form, rnd):
    """n messages signed by the key of `form`, some with h, z or the message altered"""
    pws, pubs, comb, tors = keys(d)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    if form == "torsion":
        # no password: signed the reference's way with TORSION_S, so a signature verifies iff BE(h) = 0 (mod 4) (quirk
        # Q10: V is multiplied by the unreduced h); the even items get nonces that make it verify
        h, zz = _torsion().sign_as(orc, TORSION_S, msgs, d, rnd, t=4, verifying=range(0, n, 2))
    else:
        signer = [pws[i % len(pws)] if form == "pub" else pws[0] for i in range(n)]
        h, zz = eng.ed448_sign(*pack(signer), *pack(msgs), d)
    h, zz = h.copy(), zz.copy()
    for i in range(0, n, 5):
        [lambda: h.__setitem__((i, 3), h[i, 3] ^ 1), lambda: zz.__setitem__((i, 50), zz[i, 50] ^ 0x10),
         lambda: None][i % 3]()
    for i in range(2, n, 7):
        if msgs[i]:
            msgs[i] = bytes([msgs[i][0] ^ 0x80]) + msgs[i][1:]
    return msgs, h, zz


@pytest.mark.parametrize("form", ["pub", "comb", "torsion"])
@pytest.mark.parametrize("n", [1, 127, 129, 4099])
@pytest.mark.parametrize("d", [256, 384, 512])
def test_verify_parity(eng, orc, keys, d, n, form):
    rnd = np.random.default_rng(d * 19 + n)
    msgs, h, zz = signed(eng, orc, keys, d, n, form, rnd)
    arg, pub = key_form(keys, d, form, n)
    with eng.ed448_verify_stream(arg, h, zz, d) as st:
        for pieces in plan(rnd, msgs, SQ[d], 6):
            st.update(*pack(pieces))
        rc, ok = st.final()
    assert rc == 0
    md, mo = pack(msgs)
    _, want = eng.ed448_verify(pub.reshape(-1), md, mo, h, zz, d)
    assert np.array_equal(ok, want)
    assert np.array_equal(ok, orc.verify_batch(pub.reshape(-1), md, mo, h, zz, d, threads=0))
    if n > 5:
        assert ok.any() and not ok.all()
    i = 0
    V = E.point_from_bytes(pub[i].tobytes())
    assert bool(ok[i]) == E.verify(V, msgs[i], h[i].tobytes(), zz[i].tobytes(), d)


# ---- 4. the reference KAT sizes, one byte per update --------------------------------------------------------------------
def test_kat_sizes_one_byte_per_update(eng, orc, keys):
    with open(os.path.join(HERE, "golden", "sha3_kat.json")) as f:
        kat = json.load(f)
    sizes = sorted({len(r["msg"]) // 2 for r in kat["sha3"] + kat["tagged_hash"]} | {len(r["x"]) // 2 for r in kat["kmac_xof"]})
    assert sizes
    rnd = np.random.default_rng(4)
    msgs = [rnd.bytes(L) for L in sizes]
    n, top = len(msgs), max(sizes)
    one = [[m[k:k + 1] for m in msgs] for k in range(top)]
    for d in (256, 512):
        pws = [b"pw"] * n
        nonces = rnd.bytes(512 * n)
        with eng.sponge_encrypt_stream(*pack(pws), nonces, 512, d) as st:
            ct, tag = seal(st, one)
        for i in range(n):
            assert (ct[i], tag[i].tobytes()) == oracle_sponge(orc, msgs[i], pws[i], nonces[512 * i:512 * (i + 1)], d,
                                                              B.AE_SHA3)
        _, pubs, comb, _ = keys(d)
        k = rnd.bytes(56 * n)
        st, z = eng.ed448_key_encrypt_stream(comb, k, d)
        with st:
            ct, tag = seal(st, one)
        md, mo = pack(msgs)
        want_ct, want_tag, _ = eng.ed448_key_encrypt_prepared(comb, k, md, mo, d)
        assert b"".join(ct) == want_ct.tobytes() and np.array_equal(tag, want_tag)


# ---- 5. round trip through the one-shot decryptions and the Python API -----------------------------------------------
def test_round_trip(eng, keys):
    from capycrypt_b200 import api

    rnd = np.random.default_rng(8)
    n, d = 129, 384
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [rnd.bytes(16) for _ in range(n)]
    nonces = rnd.bytes(512 * n)
    with eng.sponge_encrypt_stream(*pack(pws), nonces, 512, d, B.AE_KEM) as st:
        ct, tag = seal(st, plan(rnd, msgs, SQ[d], 4))
    out, ok = eng.sponge_decrypt(*pack(pws), nonces, 512, *pack(ct), tag, d, B.AE_KEM)
    assert ok.all() and out.tobytes() == b"".join(msgs)
    kp_pws, pubs, comb, _ = keys(d)
    st, z = eng.ed448_key_encrypt_stream(comb, rnd.bytes(56 * n), d)
    with st:
        ct, tag = seal(st, plan(rnd, msgs, SQ[d], 4))
    rc, out, ok = eng.ed448_key_decrypt(*pack([kp_pws[0]] * n), z, *pack(ct), tag, d)
    assert rc == 0 and ok.all() and out.tobytes() == b"".join(msgs)

    g = api.Gpu(eng)
    sd = api.SecParam(d)
    with g.sha3_encrypt_stream(pws, sd) as st:
        cts = [b"".join(p) for p in zip(*[st.update(pieces) for pieces in plan(rnd, msgs, SQ[d], 3)])]
        tags = st.finish()
        ms = [api.Message(msg=bytearray(c), d=sd, digest=t, sym_nonce=z) for c, t, z in zip(cts, tags, st.nonces)]
    assert g.sha3_decrypt(ms, pws) == [None] * n and [bytes(m.msg) for m in ms] == msgs
    with g.key_encrypt_stream(comb, sd, n=n) as st:
        cts = [b"".join(p) for p in zip(*[st.update(pieces) for pieces in plan(rnd, msgs, SQ[d], 3)])]
        tags = st.finish()
        ms = [api.Message(msg=bytearray(c), d=sd, digest=t, asym_nonce=z) for c, t, z in zip(cts, tags, st.asym_nonces)]
    assert g.key_decrypt(ms, [kp_pws[0]] * n) == [None] * n and [bytes(m.msg) for m in ms] == msgs
    # verify_stream: malformed signature and key lengths fail alone, like verify()
    signer = [kp_pws[0]] * n
    h, zz = eng.ed448_sign(*pack(signer), *pack(msgs), d)
    sigs = [api.Signature(h=h[i].tobytes(), z=zz[i].tobytes()) for i in range(n)]
    sigs[3] = api.Signature(h=sigs[3].h[:55], z=sigs[3].z)
    sigs[4] = None
    pk = [pubs[0].tobytes()] * n
    pk[5] = pk[5][:111]
    with g.verify_stream(sigs, pk, sd) as st:
        for pieces in plan(rnd, msgs, SQ[d], 3):
            st.update(pieces)
        res = st.finish()
    assert [type(e).__name__ if e else None for e in res[3:6]] == ["OperationError"] * 3
    assert res[4].args[0] == "SignatureNotSet" and res[3].args[0] == res[5].args[0] == "SignatureVerificationFailure"
    assert all(e is None for i, e in enumerate(res) if i not in (3, 4, 5))
    with g.verify_stream(sigs, comb, sd) as st:
        st.update(msgs)
        res = st.finish()
    assert [e is None for e in res] == [i not in (3, 4) for i in range(n)]


# ---- 6. verification failures ---------------------------------------------------------------------------------------------
def test_verify_failures(eng, keys):
    rnd = np.random.default_rng(9)
    n, d = 40, 512
    pws, pubs, comb, _ = keys(d)
    msgs = [rnd.bytes(300) for _ in range(n)]
    h, zz = eng.ed448_sign(*pack([pws[0]] * n), *pack(msgs), d)
    h, zz = h.copy(), zz.copy()
    h[1, 0] ^= 1
    zz[2, 55] ^= 1
    pub = np.tile(pubs[0], (n, 1))
    pub[4, 0] ^= 1  # off the curve
    for arg in (pub, comb):
        with eng.ed448_verify_stream(arg, h, zz, d) as st:
            pieces = [m[:150] for m in msgs]
            st.update(*pack(pieces))
            pieces = [m[150:] if i != 3 else bytes([m[150] ^ 4]) + m[151:] for i, m in enumerate(msgs)]
            st.update(*pack(pieces))
            rc, ok = st.final()
        bad = {1, 2, 3, 4} if arg is pub else {1, 2, 3}
        assert [i for i in range(n) if not ok[i]] == sorted(bad)
        assert rc == (B.ERR_BAD_POINT if arg is pub else 0)


# ---- 7. in place, _dev buffers at odd offsets, launches -------------------------------------------------------------------
def test_in_place(eng):
    rnd = np.random.default_rng(10)
    n, d = 257, 256
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [b"x"] * n
    nonces = rnd.bytes(512 * n)
    ups = plan(rnd, msgs, SQ[d], 5)
    a = eng.sponge_encrypt_stream(*pack(pws), nonces, 512, d)
    b = eng.sponge_encrypt_stream(*pack(pws), nonces, 512, d)
    with a, b:
        for pieces in ups:
            data, off = pack(pieces)
            want = a.update(data, off)
            got = b.update(data, off, out=data)
            assert got is data and np.array_equal(data, want)
        assert np.array_equal(a.final(), b.final())


@pytest.mark.parametrize("offset", [0, 1, 3])
def test_dev_guarded(eng, keys, offset):
    import torch

    rnd = np.random.default_rng(11 + offset)
    n, d = 129, 512
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    k = rnd.bytes(56 * n)
    _, pubs, comb, _ = keys(d)
    st, z = eng.ed448_key_encrypt_stream(comb, k, d)
    assert st.device_range(0) == (0, n)
    ct = [bytearray() for _ in range(n)]
    for j, pieces in enumerate(plan(rnd, msgs, SQ[d], 5)):
        data, off = pack(pieces)
        gd = Guarded(len(data), offset, data, seed=j)
        go = Guarded(8 * (n + 1), 8 * offset, off.tobytes(), seed=100 + j)
        gc = Guarded(len(data), offset + 2, seed=200 + j)
        st.update_dev(_Ptr(gd.ptr), _Ptr(go.ptr), _Ptr(gc.ptr))
        torch.cuda.synchronize()
        assert np.array_equal(gd.get(), data)
        go.get()
        c = gc.get()
        for i in range(n):
            ct[i] += c[int(off[i]):int(off[i + 1])].tobytes()
    gt = Guarded(56 * n, offset, seed=7)
    st.final_dev(_Ptr(gt.ptr))
    torch.cuda.synchronize()
    tag = gt.get().reshape(n, 56)
    st.close()
    md, mo = pack(msgs)
    want_ct, want_tag, _ = eng.ed448_key_encrypt_prepared(comb, k, md, mo, d)
    assert b"".join(bytes(c) for c in ct) == want_ct.tobytes() and np.array_equal(tag, want_tag)

    h, zz = eng.ed448_sign(*pack([keys(d)[0][0]] * n), md, mo, d)
    with eng.ed448_verify_stream(comb, h, zz, d) as vs:
        vs.update(md, mo)
        gok = Guarded(n, offset, seed=8)
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        vs.final_dev(_Ptr(gok.ptr), flag)
        torch.cuda.synchronize()
        assert gok.get().all() and int(flag.item()) == 0


def test_launches(eng, keys, tmp_path):
    rnd = np.random.default_rng(12)
    n = 300
    msgs = [rnd.bytes(int(x)) for x in rnd.integers(0, 700, size=n)]
    data, off = pack(msgs)
    for d, L in ((256, 21), (384, 19), (512, 17)):
        st = eng.sponge_encrypt_stream(*pack([b"p"] * n), rnd.bytes(512 * n), 512, d)
        ks = _kernels(lambda: st.update(data, off), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>"], ks
        ks = _kernels(lambda: st.final(), tmp_path)
        assert ks == [f"sponge_chain_kernel<{L}>"], ks
        st.close()
    _, pubs, comb, _ = keys(512)
    h, zz = eng.ed448_sign(*pack([keys(512)[0][0]] * n), data, off, 512)
    vs = eng.ed448_verify_stream(comb, h, zz, 512)
    assert _kernels(lambda: vs.update(data, off), tmp_path) == ["sponge_chain_kernel<17>"]
    ks = _kernels(lambda: vs.final(), tmp_path)
    assert ks == ["sponge_chain_kernel<17>", "verify_compare_kernel"], ks
    vs.close()


# ---- 8. isolation from the one-shot calls -----------------------------------------------------------------------------------
def test_isolation(eng, keys):
    rnd = np.random.default_rng(13)
    n, d = 1000, 512
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
    pws = [rnd.bytes(8) for _ in range(n)]
    nonces = rnd.bytes(512 * n)
    kp_pws, pubs, comb, _ = keys(d)
    k = rnd.bytes(56 * n)
    md, mo = pack(msgs)
    h, zz = eng.ed448_sign(*pack([kp_pws[0]] * n), md, mo, d)
    ae = eng.sponge_encrypt_stream(*pack(pws), nonces, 512, d)
    ke, _ = eng.ed448_key_encrypt_stream(comb, k, d)
    vs = eng.ed448_verify_stream(comb, h, zz, d)
    other = [rnd.bytes(int(x)) for x in rnd.integers(0, 5000, size=n)]
    od, oo = pack(other)
    ae_ct, ke_ct = [bytearray() for _ in range(n)], [bytearray() for _ in range(n)]
    for pieces in plan(rnd, msgs, SQ[d], 4):
        data, off = pack(pieces)
        for st, acc in ((ae, ae_ct), (ke, ke_ct)):
            c = st.update(data, off)
            for i in range(n):
                acc[i] += c[int(off[i]):int(off[i + 1])].tobytes()
        vs.update(data, off)
        # one-shot calls on the same scratch slots between the updates
        eng.sponge_encrypt(*pack(pws), nonces, 512, od, oo, d)
        eng.kmac_xof(*pack(pws), od, oo, 512, b"SKA", d)
        eng.ed448_verify_prepared(comb, od, oo, h, zz, d)
        eng.ed448_key_encrypt_prepared(comb, k, od, oo, d)
    want_ct, want_tag = eng.sponge_encrypt(*pack(pws), nonces, 512, md, mo, d)
    assert b"".join(bytes(c) for c in ae_ct) == want_ct.tobytes() and np.array_equal(ae.final(), want_tag)
    want_ct, want_tag, _ = eng.ed448_key_encrypt_prepared(comb, k, md, mo, d)
    assert b"".join(bytes(c) for c in ke_ct) == want_ct.tobytes() and np.array_equal(ke.final(), want_tag)
    rc, ok = vs.final()
    assert rc == 0 and ok.all()
    for st in (ae, ke, vs):
        st.close()


# ---- 9. errors -------------------------------------------------------------------------------------------------------------
def test_errors(eng, keys):
    lib, ctx = eng.lib, eng._ctx
    h = C.c_void_p()
    nonce = bytes(512)
    pw, po = pack([b"pw"])
    P = lambda a: a.ctypes.data  # noqa: E731
    _, pubs, comb, _ = keys(256)
    k56, hz = np.zeros(56, np.uint8), np.zeros(56, np.uint8)
    z = np.zeros(112, np.uint8)
    # D224 for every kind; bad d; bad variant
    assert lib.capy_sponge_encrypt_stream_new(ctx, 224, 0, P(pw), P(po), nonce, 512, 1, C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_key_encrypt_stream_new(ctx, 224, None, comb.handle, P(k56), 1, P(z), C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_verify_stream_new(ctx, 224, None, comb.handle, P(hz), P(hz), 1, C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_sponge_encrypt_stream_new(ctx, 300, 0, P(pw), P(po), nonce, 512, 1, C.byref(h)) == B.ERR_BAD_SECPARAM
    assert lib.capy_sponge_encrypt_stream_new(ctx, 256, 7, P(pw), P(po), nonce, 512, 1, C.byref(h)) == B.ERR_BAD_ARG
    # null pointers
    assert lib.capy_sponge_encrypt_stream_new(ctx, 256, 0, None, P(po), nonce, 512, 1, C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_sponge_encrypt_stream_new(ctx, 256, 0, P(pw), P(po), nonce, 512, 1, None) == B.ERR_BAD_ARG
    assert lib.capy_ed448_key_encrypt_stream_new(ctx, 256, None, comb.handle, P(k56), 1, None, C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_verify_stream_new(ctx, 256, None, comb.handle, None, P(hz), 1, C.byref(h)) == B.ERR_BAD_ARG
    # both or neither of pub / key
    pb = pubs[0].copy()
    assert lib.capy_ed448_key_encrypt_stream_new(ctx, 256, P(pb), comb.handle, P(k56), 1, P(z), C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_key_encrypt_stream_new(ctx, 256, None, None, P(k56), 1, P(z), C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_verify_stream_new(ctx, 256, P(pb), comb.handle, P(hz), P(hz), 1, C.byref(h)) == B.ERR_BAD_ARG
    assert lib.capy_ed448_verify_stream_new(ctx, 256, None, None, P(hz), P(hz), 1, C.byref(h)) == B.ERR_BAD_ARG
    assert not h.value
    # an off-curve key at key_encrypt creation: no stream
    bad = pubs[0].copy()
    bad[0] ^= 1
    assert lib.capy_ed448_key_encrypt_stream_new(ctx, 256, P(bad), None, P(k56), 1, P(z), C.byref(h)) == B.ERR_BAD_POINT
    assert not h.value
    with pytest.raises(B.CapyError):
        eng.ed448_key_encrypt_stream(bad, k56, 256)
    # a prepared key and streams of another ctx
    e2 = Engine()
    try:
        with pytest.raises(B.CapyError):
            e2.ed448_verify_stream(comb, hz, hz, 256)
        with pytest.raises(B.CapyError):
            e2.ed448_key_encrypt_stream(comb, k56, 256)
        st = eng.sponge_encrypt_stream(pw, po, nonce, 512, 256)
        d1, o1 = pack([b"abc"])
        ct = np.zeros(3, np.uint8)
        assert lib.capy_hasher_encrypt_update(e2._ctx, st.handle, P(d1), P(o1), P(ct)) == B.ERR_BAD_ARG
    finally:
        e2.close()
    # calls that do not match the kind
    out = np.zeros(64, np.uint8)
    assert lib.capy_hasher_update(ctx, st.handle, P(d1), P(o1)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_encrypt_update(ctx, st.handle, P(d1), P(o1), None) == B.ERR_BAD_ARG
    assert lib.capy_hasher_final(ctx, st.handle, 448, None, P(out)) == B.ERR_BAD_ARG  # sponge AE tags are 512 bits
    assert lib.capy_hasher_verify_final(ctx, st.handle, P(out)) == B.ERR_BAD_ARG
    vs = eng.ed448_verify_stream(comb, hz, hz, 256)
    assert lib.capy_hasher_final(ctx, vs.handle, 448, None, P(out)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_encrypt_update(ctx, vs.handle, P(d1), P(o1), P(ct)) == B.ERR_BAD_ARG
    with eng.sha3_hasher(1, 256) as sh:
        assert lib.capy_hasher_encrypt_update(ctx, sh.handle, P(d1), P(o1), P(ct)) == B.ERR_BAD_ARG
        assert lib.capy_hasher_verify_final(ctx, sh.handle, P(out)) == B.ERR_BAD_ARG
    # update after final
    st.update(d1, o1)
    st.final()
    assert lib.capy_hasher_encrypt_update(ctx, st.handle, P(d1), P(o1), P(ct)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_final(ctx, st.handle, 512, None, P(out)) == B.ERR_BAD_ARG
    vs.update(d1, o1)
    vs.final()
    assert lib.capy_hasher_update(ctx, vs.handle, P(d1), P(o1)) == B.ERR_BAD_ARG
    assert lib.capy_hasher_verify_final(ctx, vs.handle, P(out)) == B.ERR_BAD_ARG
    st.close()
    vs.close()
    # n == 0: streams whose calls do nothing
    e0, o0 = pack([])
    with eng.sponge_encrypt_stream(e0, o0, b"", 512, 256) as st:
        assert st.update(e0, o0).size == 0 and st.final().shape == (0, 64)


# ---- 10. scale ------------------------------------------------------------------------------------------------------------------
def test_scale_2e16_streams(eng, orc):
    """2^16 sponge-AE streams x 16 updates of 4 KiB through the _dev calls, against the one-shot call on the 64 KiB
    messages and the oracle on a seeded sample"""
    import torch

    n, d, piece, ups = 1 << 16, 512, 4096, 16
    g = torch.Generator(device="cuda").manual_seed(14)
    msgs = torch.randint(0, 256, (n, ups * piece), dtype=torch.uint8, device="cuda", generator=g)
    pws = [b"scale %d" % i for i in range(n)]
    nonces = np.random.default_rng(14).bytes(512 * n)
    pd, po = pack(pws)
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * piece
    ct = torch.empty_like(msgs)
    with eng.sponge_encrypt_stream(pd, po, nonces, 512, d) as st:
        for k in range(ups):
            src = msgs[:, k * piece:(k + 1) * piece].contiguous()
            dst = torch.empty_like(src)
            st.update_dev(src, off, dst)
            ct[:, k * piece:(k + 1) * piece] = dst
        tag = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
        st.final_dev(tag)
        torch.cuda.synchronize()
    flat = msgs.reshape(-1)
    moff = torch.arange(n + 1, dtype=torch.int64, device="cuda") * (ups * piece)
    want_ct = torch.empty_like(flat)
    want_tag = torch.empty_like(tag)
    t_pd, t_po = torch.from_numpy(pd).cuda(), torch.from_numpy(po.astype(np.int64)).cuda()
    t_nonce = torch.from_numpy(np.frombuffer(nonces, np.uint8).copy()).cuda()
    eng.sponge_encrypt_dev(t_pd, t_po, len(pd), t_nonce, 512, flat, moff, d, want_ct, want_tag)
    torch.cuda.synchronize()
    assert torch.equal(ct.reshape(-1), want_ct) and torch.equal(tag, want_tag)
    for i in np.random.default_rng(15).choice(n, 4, replace=False):
        m = msgs[i].cpu().numpy().tobytes()
        oc, ot = oracle_sponge(orc, m, pws[i], nonces[512 * i:512 * (i + 1)], d, B.AE_SHA3)
        assert ct[i].cpu().numpy().tobytes() == oc and tag[i].cpu().numpy().tobytes() == ot, i


# ---- 11. two devices ------------------------------------------------------------------------------------------------------------
def test_two_devices(orc):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    e2 = Engine([0, 1])
    try:
        rnd = np.random.default_rng(21)
        n, d = 301, 512
        msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ[d])]
        pws = [rnd.bytes(9) for _ in range(n)]
        nonces = rnd.bytes(512 * n)
        with e2.sponge_encrypt_stream(*pack(pws), nonces, 512, d) as st:
            (a0, a1), (b0, b1) = st.device_range(0), st.device_range(1)
            assert a0 == 0 and a1 == b0 and b1 == n
            ct, tag = seal(st, plan(rnd, msgs, SQ[d], 4))
        for i in range(0, n, 50):
            assert (ct[i], tag[i].tobytes()) == oracle_sponge(orc, msgs[i], pws[i], nonces[512 * i:512 * (i + 1)], d,
                                                              B.AE_SHA3)
    finally:
        e2.close()


# ---- 12. the C++ mirror -----------------------------------------------------------------------------------------------------------
def test_cpp_mirror(eng, tmp_path):
    root = os.path.dirname(HERE)
    libdir = os.path.join(root, "capycrypt_b200", "_lib")
    exe = str(tmp_path / "streams_mirror_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(HERE, "host", "streams_mirror_check.cpp"),
                    "-L" + libdir, "-lcapycrypt_gpu", "-Wl,-rpath," + os.path.abspath(libdir)], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
