"""GPU parity tests for the Ed448 path: CUDA engine (through the C ABI) vs the CPU oracle on identical
seeded inputs; bit-exact.  Mirrors the reference's own tests (tests/integration_tests.rs:20-130: sign/verify
and ECDH round trips, wrong key rejects) and adds exact-value parity against the oracle, whose arithmetic
is itself pinned by OpenSSL (tests/test_oracle_ed448.py)."""
import random

import numpy as np
import pytest

from capycrypt_b200 import pack
from capycrypt_b200 import _binding as B
from oracle import ref_ed448 as E

pytestmark = pytest.mark.gpu
R = E.R
SCALARS = [0, 1, 2, 7, 8, 9, 15, 16, R - 1, R, R + 1, 2**446 - 1, 2**448 - 1, int("8" * 112, 16), int("7" * 112, 16),
           int("f" * 112, 16), int("9" * 112, 16)]


def _be(vals):
    return np.frombuffer(b"".join(v.to_bytes(56, "big") for v in vals), dtype=np.uint8)


def test_fixed_base_edge_and_random(engine, oracle):
    rnd = random.Random(1)
    ks = SCALARS + [rnd.randrange(2**448) for _ in range(1000)]
    sc = _be(ks)
    got = engine.ed448_fixed_base(sc)
    want = oracle.fixed_base_batch(sc, threads=0)
    assert np.array_equal(got, want), np.nonzero((got != want).any(axis=1))[0][:10]
    # exact value vs the Python big-int oracle for the edge cases
    for k, row in zip(ks[:len(SCALARS)], got):
        assert row.tobytes() == E.point_to_bytes(E.scalar_mult(k % R, E.GENERATOR)), k


def test_fixed_base_openssl(engine):
    """Independent pin: RFC 8032 Ed448 public keys from OpenSSL for random seeds."""
    import hashlib

    ed448 = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.ed448")
    from cryptography.hazmat.primitives import serialization as S

    rnd = random.Random(2)
    sks = [rnd.randbytes(57) for _ in range(16)]
    ks = []
    for sk in sks:
        h = bytearray(hashlib.shake_256(sk).digest(114)[:57])
        h[0] &= 0xFC
        h[55] |= 0x80
        h[56] = 0
        ks.append(int.from_bytes(h, "little"))
    got = engine.ed448_fixed_base(_be(ks))
    for sk, row in zip(sks, got):
        pub = ed448.Ed448PrivateKey.from_private_bytes(sk).public_key().public_bytes(S.Encoding.Raw, S.PublicFormat.Raw)
        assert E.rfc8032_encode(E.point_from_bytes(row.tobytes())) == pub


def test_var_base_edge_and_random(engine, oracle):
    rnd = random.Random(3)
    pts = [E.IDENTITY, (0, E.P - 1), (1, 0), (E.P - 1, 0), E.GENERATOR, E.point_add(E.GENERATOR, (1, 0))]
    pts += [E.scalar_mult(rnd.randrange(R), E.GENERATOR) for _ in range(10)]
    ks, ps = [], []
    for pt in pts:
        for k in SCALARS + [rnd.randrange(2**448) for _ in range(8)]:
            ks.append(k)
            ps.append(E.point_to_bytes(pt))
    sc = _be(ks)
    pp = np.frombuffer(b"".join(ps), dtype=np.uint8)
    rc, got = engine.ed448_var_base(sc, pp)
    assert rc == 0
    rc2, want = oracle.var_base_batch(sc, pp, threads=0)
    assert rc2 == 0
    assert np.array_equal(got, want), np.nonzero((got != want).any(axis=1))[0][:10]
    # small-order / unreduced cases against the big-int oracle (quirk Q10: exact integer)
    for i in range(0, 6 * 25, 7):
        assert got[i].tobytes() == E.point_to_bytes(E.scalar_mult(ks[i], E.point_from_bytes(ps[i]))), i


@pytest.mark.parametrize("n", [1, 2, 31, 127, 128, 129, 257])
def test_odd_batch_sizes_hit_the_partial_last_block(engine, oracle, n):
    """The curve kernels keep idle threads of the last block in the loops (block barriers): batch sizes around the block
    size must neither hang nor touch memory past the batch."""
    rnd = random.Random(500 + n)
    sc = _be([rnd.randrange(2**448) for _ in range(n)])
    fixed = engine.ed448_fixed_base(sc)
    assert np.array_equal(fixed, oracle.fixed_base_batch(sc, threads=0))
    rc, var = engine.ed448_var_base(sc, fixed.reshape(-1))
    rc2, want = oracle.var_base_batch(sc, fixed.reshape(-1), threads=0)
    assert rc == rc2 == 0 and np.array_equal(var, want)
    pws, po = pack([rnd.randbytes(rnd.randrange(0, 40)) for _ in range(n)])
    md, mo = pack([rnd.randbytes(rnd.randrange(0, 300)) for _ in range(n)])
    h, z = engine.ed448_sign(pws, po, md, mo, 256)
    ho, zo = oracle.sign_batch(pws, po, md, mo, 256, threads=0)
    assert np.array_equal(h, ho) and np.array_equal(z, zo)
    rc, ok = engine.ed448_verify(engine.ed448_keygen(pws, po, 256), md, mo, h, z, 256)
    assert rc == 0 and ok.all()


def test_var_base_openssl_x448(engine):
    """Independent pin of the variable-base path: RFC 7748 X448 shared secrets from OpenSSL equal y^2 / x^2 of the
    engine's [k]P (edwards448 -> curve448 map of RFC 7748 4.2) for clamped scalars and random base points."""
    x448 = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.x448")
    rnd = random.Random(33)
    ks, pts, shared = [], [], []
    for _ in range(32):
        k = bytearray(rnd.randbytes(56))
        base = E.scalar_mult(rnd.randrange(1, R), E.GENERATOR)
        u = E.montgomery_u(base)
        shared.append(x448.X448PrivateKey.from_private_bytes(bytes(k)).exchange(
            x448.X448PublicKey.from_public_bytes(u.to_bytes(56, "little"))))
        k[0] &= 252
        k[55] |= 128
        ks.append(int.from_bytes(k, "little"))
        pts.append(E.point_to_bytes(base))
    rc, got = engine.ed448_var_base(_be(ks), np.frombuffer(b"".join(pts), dtype=np.uint8))
    assert rc == 0
    for row, want in zip(got, shared):
        assert E.montgomery_u(E.point_from_bytes(row.tobytes())).to_bytes(56, "little") == want


def test_var_base_rejects_off_curve_points(engine):
    good = E.point_to_bytes(E.GENERATOR)
    bad = E.point_to_bytes((5, 7))
    sc = _be([3, 3, 3])
    rc, out = engine.ed448_var_base(sc, np.frombuffer(good + bad + good, dtype=np.uint8))
    assert rc == B.ERR_BAD_POINT
    assert out[0].tobytes() == E.point_to_bytes(E.scalar_mult(3, E.GENERATOR))
    assert not out[1].any()
    assert out[2].tobytes() == out[0].tobytes()


@pytest.mark.parametrize("d", (224, 256, 384, 512))
def test_keygen(engine, oracle, d):
    rnd = random.Random(10 + d)
    pws = [b"", b"a", rnd.randbytes(130), rnd.randbytes(131), rnd.randbytes(300)] + \
          [rnd.randbytes(rnd.randrange(0, 64)) for _ in range(300)]
    pd, po = pack(pws)
    got = engine.ed448_keygen(pd, po, d)
    want = oracle.keygen_batch(pd, po, d, threads=0)
    assert np.array_equal(got, want), np.nonzero((got != want).any(axis=1))[0][:10]


@pytest.mark.parametrize("d", (256, 512))
def test_sign_verify(engine, oracle, d):
    rnd = random.Random(20 + d)
    n = 200
    pws = [rnd.randbytes(rnd.choice([0, 1, 16, 32, 100])) for _ in range(n)]
    msgs = [rnd.randbytes(rnd.choice([0, 1, 64, 135, 136, 256, 1000, 4096])) for _ in range(n)]
    pd, po = pack(pws)
    md, mo = pack(msgs)
    h, z = engine.ed448_sign(pd, po, md, mo, d)
    hw, zw = oracle.sign_batch(pd, po, md, mo, d, threads=0)
    assert np.array_equal(h, hw), np.nonzero((h != hw).any(axis=1))[0][:10]
    assert np.array_equal(z, zw), np.nonzero((z != zw).any(axis=1))[0][:10]
    pub = engine.ed448_keygen(pd, po, d)
    rc, ok = engine.ed448_verify(pub, md, mo, h, z, d)
    assert rc == 0 and ok.all()
    # the oracle accepts the engine's signatures too
    assert oracle.verify_batch(pub, md, mo, h, z, d, threads=0).all()
    # tamper: flipped h byte, flipped z byte, wrong public key, changed message
    h2 = h.copy(); h2[0, 0] ^= 1
    z2 = z.copy(); z2[1, 55] ^= 1
    rc, ok = engine.ed448_verify(pub, md, mo, h2, z2, d)
    assert rc == 0 and list(ok[:3]) == [0, 0, 1] and ok[2:].all()
    pub2 = pub.copy(); pub2[[3, 4]] = pub[[4, 3]]
    rc, ok = engine.ed448_verify(pub2, md, mo, h, z, d)
    want = oracle.verify_batch(pub2, md, mo, h, z, d, threads=0)
    assert rc == 0 and np.array_equal(ok, want) and ok[3] == 0 and ok[4] == 0
    md2 = md.copy()
    if len(md2):
        md2[int(mo[6])] ^= 0x80 if mo[7] > mo[6] else 0
    rc, ok = engine.ed448_verify(pub, md2, mo, h, z, d)
    assert np.array_equal(ok, oracle.verify_batch(pub, md2, mo, h, z, d, threads=0))


def test_verify_with_off_curve_key(engine):
    pd, po = pack([b"pw"] * 2)
    md, mo = pack([b"m1", b"m2"])
    h, z = engine.ed448_sign(pd, po, md, mo, 512)
    pub = engine.ed448_keygen(pd, po, 512)
    pub[1] = np.frombuffer(E.point_to_bytes((5, 7)), dtype=np.uint8)
    rc, ok = engine.ed448_verify(pub, md, mo, h, z, 512)
    assert rc == B.ERR_BAD_POINT and list(ok) == [1, 0]


def test_ecdh_agreement(engine, oracle):
    """ecc/encryptable.rs:36-38 vs :76-78: x([k]V) == x([s]Z) with Z = [k]G, V = [s]G."""
    rnd = random.Random(30)
    n = 64
    pws = [rnd.randbytes(16) for _ in range(n)]
    pd, po = pack(pws)
    pub = engine.ed448_keygen(pd, po, 512)
    k = np.frombuffer(rnd.randbytes(56 * n), dtype=np.uint8)
    rc, wx, Z = engine.ed448_ecdh(k, pub)
    assert rc == 0
    rc2, wx_o = oracle.ecdh_batch(k, pub, threads=0)
    assert rc2 == 0 and np.array_equal(wx, wx_o)
    # decrypt side: W' = [s]Z with s from the password
    s_be = _be([E.secret_scalar(pw, 512) for pw in pws])
    rc, W2 = engine.ed448_var_base(s_be, Z)
    assert rc == 0 and np.array_equal(W2[:, :56], wx)


def test_ecdh_without_z(engine):
    """capy_ed448_ecdh_batch with z_xy112 == NULL: the same W.x as with Z requested, and a bad point is still reported."""
    rnd = random.Random(31)
    n = 64
    pd, po = pack([rnd.randbytes(16) for _ in range(n)])
    pub = engine.ed448_keygen(pd, po, 512)
    k = np.frombuffer(rnd.randbytes(56 * n), dtype=np.uint8)
    rc, wx, Z = engine.ed448_ecdh(k, pub)
    assert rc == 0 and Z is not None
    rc, wx_only, Z_none = engine.ed448_ecdh(k, pub, want_z=False)
    assert rc == 0 and Z_none is None and np.array_equal(wx_only, wx)
    pub[5] = np.frombuffer(E.point_to_bytes((5, 7)), dtype=np.uint8)
    rc, wx_bad, _ = engine.ed448_ecdh(k, pub, want_z=False)
    keep = np.arange(n) != 5
    assert rc == B.ERR_BAD_POINT and not wx_bad[5].any() and np.array_equal(wx_bad[keep], wx[keep])


def test_unsupported_security_parameter(engine):
    pd, po = pack([b"pw"])
    with pytest.raises(B.CapyError) as e:
        engine.ed448_keygen(pd, po, 100)
    assert e.value.status == B.ERR_BAD_SECPARAM


def test_fixed_base_large_batch_properties(engine, oracle):
    """A larger batch: seeded sample vs the oracle, plus the group law [a]G + [b]G == [a+b]G checked on the
    engine's own outputs for every item (size-independent property)."""
    n = 1 << 14
    rnd = np.random.default_rng(5)
    a = rnd.integers(0, 256, size=(n, 56), dtype=np.uint8)
    got = engine.ed448_fixed_base(a.reshape(-1))
    idx = rnd.choice(n, size=256, replace=False)
    want = oracle.fixed_base_batch(np.ascontiguousarray(a[idx]).reshape(-1), threads=0)
    assert np.array_equal(got[idx], want)
    # [k]G computed as a variable-base multiplication of G must agree for every item
    G = np.tile(np.frombuffer(E.point_to_bytes(E.GENERATOR), dtype=np.uint8), n)
    rc, got_vb = engine.ed448_var_base(a.reshape(-1), G)
    assert rc == 0 and np.array_equal(got_vb, got)
