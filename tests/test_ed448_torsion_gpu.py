"""Ed448 with public keys and nonce points outside the prime-order subgroup: the unreduced h of verify (quirk Q10).

verify computes U' = [z]G + [BE(h)]V with the whole 448-bit integer BE(h), never BE(h) mod r (signable.rs:76-77).  Both
give the same point when V has order r; they differ when V = [s]G + T has a torsion component T of order t in {2, 4}.
A signature made the reference's way -- U = [k]G, h = KMACXOF(U.x, m, 448, "T", d), z = k - BE(h) s mod r -- gives
U' = U + [BE(h)]T, so it verifies iff BE(h) = 0 (mod t).  A verify that reduced h first would answer for
(BE(h) mod r) mod t instead; r = 3 (mod 4) and BE(h) >= r about 3/4 of the time, so the two rules disagree on many
messages.  ECDHIES has two such rules: key_encrypt to [s]G + T (k = 4 BE(k_rand) mod r) decrypts with the password of s
iff k = 0 (mod t), and a ciphertext whose nonce point was replaced by Z + T' decrypts iff s = 0 (mod ord T').

The generators below build signatures and ciphertexts whose expected result follows from these rules alone, with the C
oracle for [k]G and KMAC, and check the rules against the C oracle as they go.  The CPU tests check the rules against
the Python oracle too; the GPU tests hold every entry point to them."""
import ctypes as C
import functools
import importlib.util
import os
from dataclasses import dataclass

import numpy as np
import pytest

from capycrypt_b200.engine import pack
from oracle import cpu
from oracle import ref_ed448 as E

HERE = os.path.dirname(os.path.abspath(__file__))
P, R = E.P, E.R


def _load(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_S = _load("test_streams_gpu")  # the input generators, and the guarded-buffer helpers
Guarded, SQ, lengths, plan, seal = _S.Guarded, _S.SQ, _S.lengths, _S.plan, _S.seal

# ---- the points of small order and the key classes ------------------------------------------------------------------
T2 = (0, P - 1)  # order 2
T4 = (1, 0)  # order 4, [2]T4 = T2
T4N = (P - 1, 0)  # order 4, -T4
ORDER = {None: 1, T2: 2, T4: 4, T4N: 4}
NAME = {None: "O", T2: "T2", T4: "T4", T4N: "T4'"}

# (name, has a secret scalar s (else s = 0), torsion component T)
CLASSES = (("sG", True, None), ("O", False, None), ("sG+T2", True, T2), ("sG+T4", True, T4), ("sG+T4'", True, T4N),
           ("T2", False, T2), ("T4", False, T4))
NAMES = tuple(c[0] for c in CLASSES)
COMB = {"sG", "O"}  # [r]V = O: a prepared key gets a comb table


def be(x: int) -> bytes:
    return x.to_bytes(56, "big")


def rows(values) -> np.ndarray:
    """56-byte big-endian rows of integers"""
    return np.frombuffer(b"".join(be(v) for v in values), np.uint8).reshape(-1, 56).copy()


def nonce(rnd) -> int:
    return int.from_bytes(rnd.bytes(56), "big") % R


def exact_rule(h: int, t: int) -> bool:
    """U' = U + [BE(h)]T is U"""
    return h % t == 0


def reduced_rule(h: int, t: int) -> bool:
    """what a verify that multiplied V by BE(h) mod r would decide"""
    return h % R % t == 0


def multiple(j: int, T):
    """[j]T (the identity for T = None)"""
    acc = E.IDENTITY
    for _ in range(j):
        acc = E.point_add(acc, T)
    return acc


@dataclass(frozen=True)
class Key:
    name: str
    pw: bytes | None  # the password of s (None: s = 0)
    s: int
    T: tuple | None
    t: int  # the order of T
    pub: bytes  # x || y of [s]G + T


def secret_scalars(orc, pws, d) -> list[int]:
    """s = 4 * BE(KMACXOF(pw, "", 448, "SK", d)) mod r  (ecc/keypair.rs:42-43)"""
    out = orc.kmac_xof_batch(*cpu.pack(pws), *cpu.pack([b""] * len(pws)), 448, b"SK", d, threads=0)
    return [int.from_bytes(r.tobytes(), "big") * 4 % R for r in out]


def times_g(orc, scalars) -> list:
    """[k]G, affine, by the C oracle"""
    out = orc.fixed_base_batch(b"".join(be(k) for k in scalars), threads=0)
    return [E.point_from_bytes(r.tobytes()) for r in out]


def key(orc, name, pw, s, T) -> Key:
    V = times_g(orc, [s])[0] if s else E.IDENTITY
    if T is not None:
        V = E.point_add(V, T)
    return Key(name, pw, s, T, ORDER[T], E.point_to_bytes(V))


@functools.lru_cache(maxsize=None)
def keys(d: int) -> tuple[Key, ...]:
    """one key per class of CLASSES; s from a password"""
    orc = cpu.get()
    pws = [b"torsion test key " + c[0].encode() for c in CLASSES]
    ss = secret_scalars(orc, pws, d)
    return tuple(key(orc, name, pw if secret else None, s if secret else 0, T)
                 for (name, secret, T), pw, s in zip(CLASSES, pws, ss))


# ---- signatures -------------------------------------------------------------------------------------------------------
def h_of(orc, ks, msgs, d) -> list[int]:
    """BE(h) for h = KMACXOF(([k]G).x, m, 448, "T", d)  (ecc/signable.rs:48-51)"""
    if not ks:
        return []
    U = orc.fixed_base_batch(b"".join(be(k) for k in ks), threads=0)
    ko = np.arange(len(ks) + 1, dtype=np.uint64) * 56
    out = orc.kmac_xof_batch(U[:, :56].reshape(-1), ko, *cpu.pack(msgs), 448, b"T", d, threads=0)
    return [int.from_bytes(r.tobytes(), "big") for r in out]


def sign_as(orc, s, msgs, d, rnd, t=1, verifying=()):
    """(h, z) as the reference signs with the secret scalar s (ecc/signable.rs:40-57) and fresh nonces k.  The items in
    `verifying` get their nonce drawn again until BE(h) = 0 (mod t): they verify against [s]G + T for T of order t."""
    ks = [nonce(rnd) for _ in msgs]
    hs = h_of(orc, ks, msgs, d)
    todo = [i for i in verifying if hs[i] % t]
    while todo:
        for i in todo:
            ks[i] = nonce(rnd)
        for i, h in zip(todo, h_of(orc, [ks[i] for i in todo], [msgs[i] for i in todo], d)):
            hs[i] = h
        todo = [i for i in todo if hs[i] % t]
    return rows(hs), rows((k - h * s) % R for k, h in zip(ks, hs))


def requirements(t: int, slots: int):
    """(what, predicate of BE(h)) that the signatures of a key class with torsion of order t must each meet at least
    once: every residue mod 4 on both sides of r, where the exact and the reduced rule disagree (both ways), and the
    signatures that verify and become the controls (one bit of z flipped)"""
    req = [(f"BE(h) = {j} (mod 4), BE(h) {'<' if low else '>='} r", lambda h, j=j, low=low: h % 4 == j and (h < R) == low)
           for j in range(4) for low in (True, False)]
    if t > 1:
        req += [("verifies, h mod r would not", lambda h: exact_rule(h, t) and not reduced_rule(h, t)),
                ("fails, h mod r would verify", lambda h: reduced_rule(h, t) and not exact_rule(h, t))]
    return req + [("control", lambda h: exact_rule(h, t))] * max(1, slots // 32)


@dataclass
class Signed:
    d: int
    keys: tuple[Key, ...]
    cls: np.ndarray  # the key (index into keys) of every item
    msgs: list[bytes]
    hv: list[int]  # BE(h)
    h: np.ndarray  # n x 56
    z: np.ndarray  # n x 56
    control: np.ndarray  # a signature that verified, with one bit of z flipped
    want: np.ndarray  # the exact rule (0 for the controls)
    reduced: np.ndarray  # what a verify that reduced h mod r would give
    oracle: np.ndarray  # the C oracle's verify_batch

    @property
    def n(self) -> int:
        return len(self.msgs)

    @property
    def pub(self) -> np.ndarray:
        return np.frombuffer(b"".join(self.keys[c].pub for c in self.cls), np.uint8).reshape(-1, 112)

    def why(self, ok) -> list:
        """the items where ok is not the rule: key class, BE(h) mod 4, BE(h) >= r, and whether ok is the reduced rule"""
        bad = np.nonzero(np.asarray(ok) != self.want)[0]
        return [(int(i), self.keys[self.cls[i]].name, "control" if self.control[i] else self.hv[i] % 4,
                 self.hv[i] >= R, "h mod r" if ok[i] == self.reduced[i] else "") for i in bad[:12]]


def coverage(c: Signed) -> None:
    """every key class meets its requirements (a single item: the two rules disagree on it)"""
    if c.n == 1:
        assert not c.control[0] and c.want[0] != c.reduced[0]
        return
    for ci in sorted(set(c.cls.tolist())):
        items = [i for i in range(c.n) if c.cls[i] == ci]
        t = c.keys[ci].t
        for what, pred in requirements(t, len(items)):
            if what == "control":
                continue
            assert any(pred(c.hv[i]) for i in items if not c.control[i]), (c.keys[ci].name, what)
        assert any(c.control[i] for i in items), (c.keys[ci].name, "control")
        assert all(not c.want[i] for i in items if c.control[i])


def signed(d: int, n: int, names: tuple[str, ...] = NAMES) -> Signed:
    """n signatures over seeded messages (lengths with the block edges) by the key classes `names`, mixed.  The nonces are
    drawn again until every class meets requirements(); n = 1: one signature by sG+T4 that verifies while the reduced
    rule rejects it."""
    return _signed(d, n, tuple(names))


@functools.lru_cache(maxsize=None)
def _signed(d: int, n: int, names: tuple[str, ...]) -> Signed:
    orc = cpu.get()
    rnd = np.random.default_rng([d, n] + [NAMES.index(x) for x in names])
    ks_all = keys(d)
    use = [NAMES.index(x) for x in names]
    if n == 1:
        use = [NAMES.index("sG+T4")]
    cls = np.array(use)[rnd.permutation(np.arange(n) % len(use))]
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ.get(d, 172))]
    ks = [nonce(rnd) for _ in range(n)]
    hv = h_of(orc, ks, msgs, d)
    slots = {ci: [i for i in range(n) if cls[i] == ci] for ci in use}
    if n == 1:
        need = {use[0]: [r for r in requirements(4, 1) if r[0] == "verifies, h mod r would not"]}
    else:
        need = {ci: requirements(ks_all[ci].t, len(slots[ci])) for ci in use}
        for ci in use:
            assert len(need[ci]) <= len(slots[ci]), f"{len(slots[ci])} items of {NAMES[ci]} cannot meet its requirements"
    taken, role = set(), {}
    for _ in range(200):
        for ci in use:
            left = []
            for what, pred in need[ci]:
                i = next((i for i in slots[ci] if i not in taken and pred(hv[i])), None)
                if i is None:
                    left.append((what, pred))
                else:
                    taken.add(i)
                    role[i] = what
            need[ci] = left
        if not any(need.values()):
            break
        redraw = []  # new nonces for some free items of the classes that still miss something
        for ci in use:
            if need[ci]:
                free = [i for i in slots[ci] if i not in taken]
                redraw += [free[j] for j in sorted(rnd.permutation(len(free))[:64])]
        for i in redraw:
            ks[i] = nonce(rnd)
        for i, h in zip(redraw, h_of(orc, [ks[i] for i in redraw], [msgs[i] for i in redraw], d)):
            hv[i] = h
    assert not any(need.values()), need
    z = rows((k - h * ks_all[c].s) % R for k, h, c in zip(ks, hv, cls))
    control = np.array([role.get(i) == "control" for i in range(n)])
    for i in np.nonzero(control)[0]:
        z[i, int(rnd.integers(0, 56))] ^= 1 << int(rnd.integers(0, 8))
    t = [ks_all[c].t for c in cls]
    want = np.array([exact_rule(h, tt) and not f for h, tt, f in zip(hv, t, control)], np.uint8)
    reduced = np.array([reduced_rule(h, tt) and not f for h, tt, f in zip(hv, t, control)], np.uint8)
    c = Signed(d, ks_all, cls, msgs, hv, rows(hv), z, control, want, reduced, None)
    md, mo = cpu.pack(msgs)
    c.oracle = orc.verify_batch(c.pub, md, mo, c.h, c.z, d, threads=0)
    assert np.array_equal(c.oracle, c.want), c.why(c.oracle)
    coverage(c)
    return c


# ---- ECDHIES ----------------------------------------------------------------------------------------------------------
def oracle_key_encrypt(orc, pub, k_rand, msgs, d):
    """(ct, tag, Z) of KeyEncryptable::key_encrypt (ecc/encryptable.rs:34-50) with the C oracle's ECDH and KMACXOF"""
    rc, wx = orc.ecdh_batch(k_rand, pub, threads=0)
    assert rc == 0
    z = orc.fixed_base_batch(rows(int.from_bytes(k.tobytes(), "big") * 4 % R for k in k_rand), threads=0)
    ct, tag = seal_with(orc, wx, msgs, d)
    return ct, tag, z


def _keymat(orc, wx, d):
    n = len(wx)
    ko = np.arange(n + 1, dtype=np.uint64) * 56
    km = orc.kmac_xof_batch(wx.reshape(-1), ko, *cpu.pack([b""] * n), 896, b"PK", d, threads=0)
    return km[:, :56].copy(), km[:, 56:].copy(), ko


def _keystream(orc, ke, ko, lens, d):
    """KMACXOF(ke, "", 8 L, "PKE"): one long squeeze cut to every length (the output of KMACXOF does not depend on L)"""
    n = len(lens)
    top = max(list(lens) + [1])
    return orc.kmac_xof_batch(ke.reshape(-1), ko, *cpu.pack([b""] * n), 8 * top, b"PKE", d, threads=0)


def seal_with(orc, wx, msgs, d):
    ke, ka, ko = _keymat(orc, wx, d)
    tag = orc.kmac_xof_batch(ka.reshape(-1), ko, *cpu.pack(msgs), 448, b"PKA", d, threads=0)
    ks = _keystream(orc, ke, ko, [len(m) for m in msgs], d)
    return [bytes(a ^ b for a, b in zip(m, ks[i].tobytes())) for i, m in enumerate(msgs)], tag


def oracle_key_decrypt(orc, pws, z, cts, tags, d):
    """(ok, buffer) of KeyEncryptable::key_decrypt (:72-94): W = [s]Z is the oracle's ECDH of KMACXOF(pw, "", 448, "SK")"""
    n = len(cts)
    sk = orc.kmac_xof_batch(*cpu.pack(pws), *cpu.pack([b""] * n), 448, b"SK", d, threads=0)
    rc, wx = orc.ecdh_batch(sk, z, threads=0)
    assert rc == 0
    ke, ka, ko = _keymat(orc, wx, d)
    ks = _keystream(orc, ke, ko, [len(c) for c in cts], d)
    pts = [bytes(a ^ b for a, b in zip(c, ks[i].tobytes())) for i, c in enumerate(cts)]
    t_new = orc.kmac_xof_batch(ka.reshape(-1), ko, *cpu.pack(pts), 448, b"PKA", d, threads=0)
    ok = np.array([t_new[i].tobytes() == tags[i].tobytes() for i in range(n)], np.uint8)
    return ok, [p if o else c for p, c, o in zip(pts, cts, ok)]


@dataclass
class Sealed:
    d: int
    what: list[str]  # per item: the recipient's key class, or "s=j mod 4, Z+T'" for a moved nonce
    t: list[int]  # the order of the torsion component of the recipient's key
    pub: np.ndarray  # n x 112
    k_rand: np.ndarray  # n x 56
    msgs: list[bytes]
    ct: list[bytes]  # the C oracle's key_encrypt
    tag: np.ndarray
    z: np.ndarray
    pws: list[bytes]  # the recipients' passwords
    want: np.ndarray  # key_decrypt with Z: k = 0 (mod t)
    z_moved: np.ndarray  # Z + T' on the items of a recipient [s]G, Z elsewhere
    want_moved: np.ndarray  # s = 0 (mod ord T') there, `want` elsewhere

    @property
    def n(self) -> int:
        return len(self.msgs)


@functools.lru_cache(maxsize=None)
def sealed(d: int, n: int) -> Sealed:
    """n key_encrypts: the even items to the keys with a password (sG, sG+T2, sG+T4, sG+T4'), with k_rand drawn so that
    k mod 4 takes every value for every key; the odd items to [s_j]G for four passwords with s_j = j (mod 4), whose
    nonce point is then moved by T2, T4 or T4'"""
    orc = cpu.get()
    rnd = np.random.default_rng([d, n, 4])
    recipients = [k for k in keys(d) if k.pw is not None]
    cands = [b"recipient %d" % i for i in range(64)]
    by_residue = {}
    for pw, s in zip(cands, secret_scalars(orc, cands, d)):
        by_residue.setdefault(s % 4, (pw, s))
    assert sorted(by_residue) == [0, 1, 2, 3]
    prime = [key(orc, f"s={j} mod 4", *by_residue[j], None) for j in range(4)]
    moves = [(kp, T) for kp in prime for T in (T2, T4, T4N)]
    what, pubs, pws, kr, moved = [], [], [], [], []
    for i in range(n):
        if i % 2 == 0:
            kp, T, k_res = recipients[(i // 2) % len(recipients)], None, (i // 2 // len(recipients)) % 4
        else:
            (kp, T), k_res = moves[(i // 2) % len(moves)], None
        while True:
            k = rnd.bytes(56)
            if k_res is None or int.from_bytes(k, "big") * 4 % R % 4 == k_res:
                break
        what.append(kp.name if T is None else f"{kp.name}, Z+{NAME[T]}")
        pubs.append(kp.pub)
        pws.append(kp.pw)
        kr.append(k)
        moved.append((kp, T))
    pub = np.frombuffer(b"".join(pubs), np.uint8).reshape(n, 112)
    k_rand = np.frombuffer(b"".join(kr), np.uint8).reshape(n, 56)
    msgs = [rnd.bytes(L) for L in lengths(rnd, n, SQ.get(d, 172))]
    ct, tag, z = oracle_key_encrypt(orc, pub, k_rand, msgs, d)
    kk = [int.from_bytes(k, "big") * 4 % R for k in kr]
    want = np.array([k % kp.t == 0 for k, (kp, _) in zip(kk, moved)], np.uint8)
    z_moved = z.copy()
    want_moved = want.copy()
    for i, (kp, T) in enumerate(moved):
        if T is not None:
            z_moved[i] = np.frombuffer(E.point_to_bytes(E.point_add(E.point_from_bytes(z[i].tobytes()), T)), np.uint8)
            want_moved[i] = kp.s % ORDER[T] == 0
    e = Sealed(d, what, [kp.t for kp, _ in moved], pub, k_rand, msgs, ct, tag, z, pws, want, z_moved, want_moved)
    # coverage: every k mod 4 for every key with a password, every (s mod 4, T') for the moved nonces
    for kp in recipients:
        assert {kk[i] % 4 for i in range(0, n, 2) if e.what[i] == kp.name} == {0, 1, 2, 3}, kp.name
    assert {e.what[i] for i in range(1, n, 2)} == {f"{kp.name}, Z+{NAME[T]}" for kp, T in moves}
    for zz, w in ((z, want), (z_moved, want_moved)):
        ok, out = oracle_key_decrypt(orc, pws, zz, ct, tag, d)
        assert np.array_equal(ok, w), [(e.what[i], int(ok[i])) for i in np.nonzero(ok != w)[0][:8]]
        assert all(out[i] == (msgs[i] if w[i] else ct[i]) for i in range(n))
    assert want.any() and not want.all() and want_moved.any() and not want_moved.all()
    return e


# ---- the batches the GPU tests use ----------------------------------------------------------------------------------
VERIFY_D, VERIFY_N = (224, 256, 384, 512), (1, 127, 129, 4099)
STREAM_D = (256, 384, 512)
PREPARED_D = (256, 512)
CLASS_N = 129  # a batch of one key class
API_D, SEALED_D, SEALED_N, DEV_D = 384, (256, 512), 129, 512


def gpu_batches():
    yield from ((d, n, NAMES) for d in VERIFY_D for n in VERIFY_N)
    yield from ((d, CLASS_N, (x,)) for d in sorted(set(PREPARED_D) | set(STREAM_D)) for x in NAMES)


# =====================================================================================================================
# CPU: the premise of the GPU tests
# =====================================================================================================================
def test_small_order_points():
    for T, t in ((T2, 2), (T4, 4), (T4N, 4)):
        assert E.on_curve(T)
        assert [multiple(j, T) == E.IDENTITY for j in range(1, t + 1)] == [False] * (t - 1) + [True]
    assert multiple(2, T4) == multiple(2, T4N) == T2 and E.point_add(T4, T4N) == E.IDENTITY
    assert R % 4 == 3


@pytest.mark.parametrize("d", [256, 512])
def test_keys_on_curve_and_orders(d):
    for k in keys(d):
        V = E.point_from_bytes(k.pub)
        assert E.on_curve(V)
        assert (E.scalar_mult(R, V) == E.IDENTITY) == (k.name in COMB), k.name
        assert (k.t == 1) == (k.name in COMB)


def test_signed_corpus_follows_the_oracles():
    """d = 256: the exact rule is what the C and the Python oracle decide, for a witness of every requirement of every
    class and for the controls; the reduced rule is not"""
    d = 256
    c = signed(d, 127)
    assert np.array_equal(c.oracle, c.want)
    assert (c.want != c.reduced).sum() >= 10
    sample = set()
    for ci in set(c.cls.tolist()):
        items = [i for i in range(c.n) if c.cls[i] == ci]
        for what, pred in requirements(c.keys[ci].t, len(items)):
            sample.add(next(i for i in items if pred(c.hv[i]) and (what == "control") == c.control[i]))
    for i in sorted(sample):
        V = E.point_from_bytes(c.keys[c.cls[i]].pub)
        assert E.verify(V, c.msgs[i], c.h[i].tobytes(), c.z[i].tobytes(), d) == bool(c.want[i]), (i, c.keys[c.cls[i]].name)
    one = signed(d, 1)
    assert one.want[0] and not one.reduced[0]
    assert E.verify(E.point_from_bytes(one.keys[one.cls[0]].pub), one.msgs[0], one.h[0].tobytes(), one.z[0].tobytes(), d)


def test_every_gpu_batch_meets_the_coverage():
    """the generator asserts coverage and the C oracle for every batch it makes: make every batch the GPU tests use"""
    for d, n, names in gpu_batches():
        coverage(signed(d, n, names))
    for d in SEALED_D:
        sealed(d, SEALED_N)


def test_sealed_corpus_follows_the_oracles():
    """d = 256: key_encrypt and key_decrypt of the Python oracle agree with the C oracle and the two ECDHIES rules"""
    d = 256
    e = sealed(d, SEALED_N)
    seen = set()
    for i in range(e.n):
        kk = int.from_bytes(e.k_rand[i].tobytes(), "big") * 4 % R
        tag = (e.what[i], kk % 4 if i % 2 == 0 else None)
        if tag in seen:
            continue
        seen.add(tag)
        if len(seen) % 5 == 1:
            c, t, Z = E.key_encrypt(E.point_from_bytes(e.pub[i].tobytes()), e.msgs[i], d, e.k_rand[i].tobytes())
            assert (c, t, E.point_to_bytes(Z)) == (e.ct[i], e.tag[i].tobytes(), e.z[i].tobytes())
        for zz, w in ((e.z, e.want), (e.z_moved, e.want_moved)):
            Z = E.point_from_bytes(zz[i].tobytes())
            assert E.key_decrypt(e.pws[i], e.ct[i], d, Z, e.tag[i].tobytes()) == \
                (bool(w[i]), e.msgs[i] if w[i] else e.ct[i]), (e.what[i], tag)
    assert len(seen) == 4 * 4 + 12


# =====================================================================================================================
# GPU
# =====================================================================================================================
def _stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def follows(c: Signed, ok) -> None:
    assert np.array_equal(ok, c.want), c.why(ok)
    assert np.array_equal(ok, c.oracle)


# ---- 1. one-shot verify, every key class in one batch -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", VERIFY_N)
@pytest.mark.parametrize("d", VERIFY_D)
def test_verify_batch(engine, d, n):
    c = signed(d, n)
    rc, ok = engine.ed448_verify(c.pub, *pack(c.msgs), c.h, c.z, d)
    assert rc == 0
    follows(c, ok)


# ---- 2. the _dev twin through guarded buffers at odd offsets -------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [1, 3])
def test_verify_batch_dev_guarded(engine, offset):
    import torch

    d = DEV_D
    c = signed(d, CLASS_N, ("sG+T4",)) if offset == 3 else signed(d, 129)
    n = c.n
    md, mo = pack(c.msgs)
    g_pub, g_m = Guarded(112 * n, offset, c.pub, seed=1), Guarded(len(md), offset, md, seed=2)
    g_off = Guarded(8 * (n + 1), 8 * offset, mo, seed=3)
    g_h, g_z = Guarded(56 * n, offset, c.h, seed=4), Guarded(56 * n, offset + 2, c.z, seed=5)
    g_ok = Guarded(n, offset, seed=6)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    engine._check(engine.lib.capy_ed448_verify_batch_dev(engine._ctx, 0, _stream(), d, g_pub.ptr, g_m.ptr, g_off.ptr, g_h.ptr,
                                                         g_z.ptr, n, g_ok.ptr, flag.data_ptr()))
    torch.cuda.synchronize()
    follows(c, g_ok.get())
    assert int(flag.item()) == 0
    for g, want in ((g_pub, c.pub), (g_m, md), (g_h, c.h), (g_z, c.z)):
        assert np.array_equal(g.get(), np.asarray(want).reshape(-1))
    g_off.get()


# ---- 3. prepared keys: the comb for sG and O, the variable-base fallback for the rest ------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("d", PREPARED_D)
def test_verify_prepared(engine, d, name):
    import torch

    c = signed(d, CLASS_N, (name,))
    n = c.n
    md, mo = pack(c.msgs)
    with engine.ed448_pub_prepare(c.keys[c.cls[0]].pub) as key:
        assert key.uses_comb == (name in COMB)
        follows(c, engine.ed448_verify_prepared(key, md, mo, c.h, c.z, d))
        g_m, g_h, g_z = Guarded(len(md), 1, md, seed=7), Guarded(56 * n, 1, c.h, seed=8), Guarded(56 * n, 3, c.z, seed=9)
        g_ok = Guarded(n, 1, seed=10)
        t_off = torch.from_numpy(mo.astype(np.int64)).cuda()
        engine._check(engine.lib.capy_ed448_verify_prepared_batch_dev(engine._ctx, 0, _stream(), d, key.handle, g_m.ptr,
                                                                      t_off.data_ptr(), g_h.ptr, g_z.ptr, n, g_ok.ptr))
        torch.cuda.synchronize()
        follows(c, g_ok.get())


# ---- 4. verify streams ---------------------------------------------------------------------------------------------------
def _stream_ok(engine, c, arg, seed):
    with engine.ed448_verify_stream(arg, c.h, c.z, c.d) as st:
        for pieces in plan(np.random.default_rng(seed), c.msgs, SQ[c.d], 6):
            st.update(*pack(pieces))
        return st.final()


@pytest.mark.gpu
@pytest.mark.parametrize("n", VERIFY_N)
@pytest.mark.parametrize("d", STREAM_D)
def test_verify_stream_per_item_keys(engine, d, n):
    c = signed(d, n)
    rc, ok = _stream_ok(engine, c, c.pub, d + n)
    assert rc == 0
    follows(c, ok)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("d", STREAM_D)
def test_verify_stream_prepared(engine, d, name):
    c = signed(d, CLASS_N, (name,))
    with engine.ed448_pub_prepare(c.keys[c.cls[0]].pub) as key:
        assert key.uses_comb == (name in COMB)
        rc, ok = _stream_ok(engine, c, key, d)
    assert rc == 0
    follows(c, ok)


# ---- 5. the Python API ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_python_api(engine):
    from capycrypt_b200.api import Gpu, Message, SecParam, Signature

    d = API_D
    gpu = Gpu(engine)
    sd = SecParam(d)

    def kinds(res):
        return [e.kind if e else None for e in res]

    def expected(c, idx):
        return [None if c.want[i] else "SignatureVerificationFailure" for i in idx]

    def sigs(c, idx):
        return [Signature(h=c.h[i].tobytes(), z=c.z[i].tobytes()) for i in idx]

    def messages(c, idx):
        return [Message(msg=bytearray(c.msgs[i]), d=sd, sig=s) for i, s in zip(idx, sigs(c, idx))]

    c = signed(d, 129)
    every = range(c.n)
    pubs = [r.tobytes() for r in c.pub]
    assert kinds(gpu.verify(messages(c, every), pubs)) == expected(c, every)
    with gpu.verify_stream(sigs(c, every), pubs, sd) as st:
        for pieces in plan(np.random.default_rng(5), c.msgs, SQ[d], 4):
            st.update(pieces)
        assert kinds(st.finish()) == expected(c, every)
    for ci in sorted(set(c.cls.tolist())):
        idx = [i for i in every if c.cls[i] == ci]
        with gpu.prepare_public_key(c.keys[ci].pub) as key:
            assert kinds(gpu.verify_prepared(messages(c, idx), key)) == expected(c, idx), c.keys[ci].name
            with gpu.verify_stream(sigs(c, idx), key, sd) as st:
                st.update([c.msgs[i] for i in idx])
                assert kinds(st.finish()) == expected(c, idx), c.keys[ci].name


# ---- 6. ECDHIES to keys with a torsion component, and nonce points with one -------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", SEALED_D)
def test_key_encrypt_to_torsion_keys(engine, d):
    e = sealed(d, SEALED_N)
    md, mo = pack(e.msgs)
    rc, ct, tag, z = engine.ed448_key_encrypt(e.pub, e.k_rand, md, mo, d)
    assert rc == 0
    assert ct.tobytes() == b"".join(e.ct) and np.array_equal(tag, e.tag) and np.array_equal(z, e.z)
    for pub in sorted({r.tobytes() for r in e.pub}):
        idx = [i for i in range(e.n) if e.pub[i].tobytes() == pub]
        with engine.ed448_pub_prepare(pub) as key:
            assert key.uses_comb == (e.t[idx[0]] == 1)
            p_ct, p_tag, p_z = engine.ed448_key_encrypt_prepared(key, e.k_rand[idx], *pack([e.msgs[i] for i in idx]), d)
        assert p_ct.tobytes() == b"".join(e.ct[i] for i in idx), e.what[idx[0]]
        assert np.array_equal(p_tag, e.tag[idx]) and np.array_equal(p_z, e.z[idx])
    st, sz = engine.ed448_key_encrypt_stream(e.pub, e.k_rand, d)
    with st:
        s_ct, s_tag = seal(st, plan(np.random.default_rng(d), e.msgs, SQ[d], 5))
    assert s_ct == e.ct and np.array_equal(s_tag, e.tag) and np.array_equal(sz, e.z)


@pytest.mark.gpu
@pytest.mark.parametrize("moved", [False, True])
@pytest.mark.parametrize("d", SEALED_D)
def test_key_decrypt_rules(engine, d, moved):
    e = sealed(d, SEALED_N)
    z, want = (e.z_moved, e.want_moved) if moved else (e.z, e.want)
    expect = [m if w else c for m, c, w in zip(e.msgs, e.ct, want)]

    def why(ok):
        return [(i, e.what[i], int(ok[i])) for i in np.nonzero(np.asarray(ok) != want)[0][:12]]

    cd, co = pack(e.ct)
    rc, out, ok = engine.ed448_key_decrypt(*pack(e.pws), z, cd, co, e.tag, d)
    assert rc == 0
    assert np.array_equal(ok, want), why(ok)
    assert out.tobytes() == b"".join(expect)
    rnd = np.random.default_rng(d + moved)
    with engine.ed448_key_decrypt_stream(*pack(e.pws), z, e.tag, d) as st:
        for pieces in plan(rnd, e.ct, SQ[d], 4):
            st.update(*pack(pieces))
        rc1, verdict = st.next_pass()
        verdict = verdict.copy()
        got = [bytearray() for _ in range(e.n)]
        for pieces in plan(rnd, e.ct, SQ[d], 5):
            data, off = pack(pieces)
            o = st.decrypt(data, off)
            for i in range(e.n):
                got[i] += o[int(off[i]):int(off[i + 1])].tobytes()
        rc2, ok2 = st.final()
    assert rc1 == rc2 == 0
    assert np.array_equal(verdict, want) and np.array_equal(ok2, want), why(ok2)
    assert [bytes(g) for g in got] == expect


# ---- 7. the kernel underneath: [k](Q + T) = [k mod r]Q + [k mod t]T ---------------------------------------------------------
@pytest.mark.gpu
def test_var_base_referee(engine, oracle):
    c = signed(256, 127)
    special = [R, R + 1, 4 * R - 1, 2**446, 2**448 - 1]
    items = [(c.hv[i], c.keys[c.cls[i]]) for i in range(c.n)] + [(k, kp) for k in special for kp in c.keys]
    ks = [k for k, _ in items]
    rc, got = engine.ed448_var_base(rows(ks), np.frombuffer(b"".join(kp.pub for _, kp in items), np.uint8))
    assert rc == 0
    sg = {kp.name: E.point_to_bytes(times_g(oracle, [kp.s])[0] if kp.s else E.IDENTITY) for kp in c.keys}  # Q = [s]G
    q = [sg[kp.name] for _, kp in items]
    orc_rc, kq = oracle.var_base_batch(rows(k % R for k in ks), np.frombuffer(b"".join(q), np.uint8), threads=0)
    assert orc_rc == 0
    table = {(NAME[T], j): multiple(j, T) for T, t in ORDER.items() for j in range(t)}
    want = [E.point_to_bytes(E.point_add(E.point_from_bytes(kq[i].tobytes()), table[NAME[kp.T], k % kp.t]))
            for i, (k, kp) in enumerate(items)]
    bad = [(i, items[i][1].name, hex(items[i][0] >> 440)) for i in range(len(items)) if got[i].tobytes() != want[i]]
    assert not bad, bad[:12]
