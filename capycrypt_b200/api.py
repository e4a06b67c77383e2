"""Host-side mirror of capyCRYPT's operator surface for BATCHES (the `capycrypt::gpu` module of the
north star, in Python because the image has no Rust toolchain; the C++ twin is host/capycrypt_gpu.hpp).

Same names, argument meaning and error behaviour as the reference:
  SecParam                      src/lib.rs:113-135      (try_from -> UnsupportedSecurityParameter)
  Message, Signature            src/lib.rs:65-94, src/ecc/signable.rs:17-24
  KeyPair::new                  src/ecc/keypair.rs:41-51
  SpongeHashable                src/sha3/hashable.rs:7-36   compute_sha3_hash / compute_tagged_hash
  Signable                      src/ecc/signable.rs:12-15   sign / verify
  kmac_xof                      src/sha3/shake_functions.rs:79-89
  SpongeEncryptable             src/sha3/encryptable.rs:7-10  sha3_encrypt / sha3_decrypt
  KeyEncryptable                src/ecc/encryptable.rs:10-13  key_encrypt / key_decrypt
Every function forwards to the CUDA engine through the C ABI; nothing is computed on the CPU.
All operations work IN PLACE on the Message objects, like the reference.
"""
from __future__ import annotations

import datetime
import os
from dataclasses import dataclass, field
from enum import IntEnum
from typing import Optional, Sequence

import numpy as np

from ._binding import ERR_BAD_POINT, CapyError
from .engine import Engine, Hasher, PreparedPublicKey, pack


class OperationError(Exception):
    """src/lib.rs:9-30 -- the variant name is carried in `.kind`."""

    def __init__(self, kind: str):
        super().__init__(kind)
        self.kind = kind


class SecParam(IntEnum):
    D224 = 224
    D256 = 256
    D384 = 384
    D512 = 512

    @staticmethod
    def try_from(value: int) -> "SecParam":
        """src/lib.rs:126-134."""
        try:
            return SecParam(value)
        except ValueError:
            raise OperationError("UnsupportedSecurityParameter") from None

    def bit_length_(self) -> int:
        return int(self)


@dataclass
class Signature:
    """src/ecc/signable.rs:17-24: h = keyed hash (56 bytes), z = scalar (56 bytes big-endian, canonical)."""
    h: bytes
    z: bytes


@dataclass
class Message:
    """src/lib.rs:65-94."""
    msg: bytearray
    d: Optional[SecParam] = None
    sym_nonce: Optional[bytes] = None
    asym_nonce: Optional[bytes] = None  # affine point x || y (112 bytes)
    digest: bytes = b""
    sig: Optional[Signature] = None
    kem_ciphertext: Optional[bytes] = b""

    @staticmethod
    def new(data: bytes) -> "Message":
        return Message(msg=bytearray(data))


@dataclass
class KeyPair:
    """src/ecc/keypair.rs:13-22.  pub_key is the affine point x || y (112 bytes LE); priv_key is the password."""
    owner: str
    pub_key: bytes
    priv_key: bytes
    date_created: str = field(default_factory=lambda: datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S"))


class Gpu:
    """`capycrypt::gpu`: batch entry points over one engine context."""

    def __init__(self, engine: Optional[Engine] = None, devices=None):
        self.engine = engine or Engine(devices)

    # ---- SpongeHashable --------------------------------------------------------------------------
    def compute_sha3_hash(self, msgs: Sequence[Message], d: SecParam, mutate_like_reference: bool = False) -> None:
        """Batched Message::compute_sha3_hash: sets every `.digest`.  With mutate_like_reference the suffix and
        padding are also appended to `.msg` as the reference does (quirk Q5, shake_functions.rs:24-29)."""
        d = SecParam.try_from(int(d))
        data, off = pack([m.msg for m in msgs])
        out = self.engine.sha3(data, off, int(d))
        for m, row in zip(msgs, out):
            m.digest = row.tobytes()
            if mutate_like_reference:
                _append_reference_padding(m.msg, int(d))

    def compute_tagged_hash(self, msgs: Sequence[Message], pws: Sequence[bytes], s: str | bytes, d: SecParam) -> None:
        d = SecParam.try_from(int(d))
        s = s.encode() if isinstance(s, str) else s
        kd, ko = pack(pws)
        xd, xo = pack([m.msg for m in msgs])
        out = self.engine.kmac_xof(kd, ko, xd, xo, int(d), s, int(d))
        for m, row in zip(msgs, out):
            m.digest = row.tobytes()

    def kmac_xof(self, keys: Sequence[bytes], xs: Sequence[bytes], l: int, s: str | bytes, d: SecParam) -> list[bytes]:
        d = SecParam.try_from(int(d))
        s = s.encode() if isinstance(s, str) else s
        kd, ko = pack(keys)
        xd, xo = pack(xs)
        return [r.tobytes() for r in self.engine.kmac_xof(kd, ko, xd, xo, l, s, int(d))]

    # ---- messages in pieces ----------------------------------------------------------------------------
    def sha3_stream(self, n: int, d: SecParam) -> "SpongeStream":
        """n compute_sha3_hash streams fed in pieces: finish() gives the digests of the concatenated pieces."""
        d = SecParam.try_from(int(d))
        return SpongeStream(self.engine.sha3_hasher(n, int(d)), int(d))

    def kmac_xof_stream(self, keys: Sequence[bytes], s: str | bytes, d: SecParam) -> "SpongeStream":
        """one kmac_xof stream per key, fed in pieces: finish(l) gives kmac_xof(key, concatenated pieces, l, s, d);
        compute_tagged_hash is finish(d).  D224 is refused (ValueError): see capy_gpu.h."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("kmac_xof_stream: D224 is not resumable (quirk Q7)")
        s = s.encode() if isinstance(s, str) else s
        kd, ko = pack(keys)
        return SpongeStream(self.engine.kmac_xof_hasher(kd, ko, s, int(d)), int(d))

    def sha3_encrypt_stream(self, pws: Sequence[bytes], d: SecParam,
                            nonces: Optional[Sequence[bytes]] = None) -> "EncryptStream":
        """one sha3_encrypt per password whose plaintext arrives in pieces: update() returns the ciphertext pieces,
        finish() the tags; together they are the .msg and .digest sha3_encrypt gives for the concatenated plaintext, and
        .nonces its .sym_nonce.  D224 is refused (ValueError): see capy_gpu.h."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("sha3_encrypt_stream: D224 is not resumable (quirk Q7)")
        if nonces is None:
            nonces = [os.urandom(512) for _ in pws]
        if len(nonces) != len(pws) or any(len(z) != 512 for z in nonces):
            raise ValueError("sha3_encrypt_stream: one 512-byte nonce per password")
        pd, po = pack(pws)
        st = self.engine.sponge_encrypt_stream(pd, po, b"".join(nonces), 512, int(d))
        return EncryptStream(st, nonces=[bytes(z) for z in nonces])

    def key_encrypt_stream(self, pub_keys: Sequence[bytes] | PreparedPublicKey, d: SecParam,
                           k_rand: Optional[Sequence[bytes]] = None, n: Optional[int] = None) -> "EncryptStream":
        """one key_encrypt per recipient (or n to one prepared key) whose plaintext arrives in pieces: as
        sha3_encrypt_stream, with .asym_nonces the Z of each message.  OperationError("InvalidPublicKey") for an
        off-curve key; D224 is refused (ValueError)."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("key_encrypt_stream: D224 is not resumable (quirk Q7)")
        prepared = isinstance(pub_keys, PreparedPublicKey)
        if n is None:
            n = len(k_rand) if k_rand is not None else (None if prepared else len(pub_keys))
        if n is None:
            raise ValueError("key_encrypt_stream: a prepared key needs n or k_rand")
        if k_rand is None:
            k_rand = [os.urandom(56) for _ in range(n)]
        if len(k_rand) != n or any(len(k) != 56 for k in k_rand):
            raise ValueError("key_encrypt_stream: one 56-byte nonce per message")
        if not prepared and (len(pub_keys) != n or any(len(p) != 112 for p in pub_keys)):
            raise ValueError("key_encrypt_stream: one 112-byte public key per message")
        pub = pub_keys if prepared else b"".join(pub_keys)
        try:
            st, z = self.engine.ed448_key_encrypt_stream(pub, b"".join(k_rand), int(d))
        except CapyError as e:
            if e.status == ERR_BAD_POINT:
                raise OperationError("InvalidPublicKey") from None
            raise
        return EncryptStream(st, asym_nonces=[r.tobytes() for r in z])

    def verify_stream(self, sigs: Sequence[Optional[Signature]], pub_keys: Sequence[bytes] | PreparedPublicKey,
                      d: SecParam) -> "VerifyStream":
        """verify() of signatures whose messages arrive in pieces: update() appends one piece per message, finish() gives
        what verify() gives for the concatenated pieces.  A missing signature (SignatureNotSet) or a malformed signature
        or key (SignatureVerificationFailure) fails on its own.  D224 is refused (ValueError)."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("verify_stream: D224 is not resumable (quirk Q7)")
        prepared = isinstance(pub_keys, PreparedPublicKey)
        res: list[Optional[OperationError]] = [None] * len(sigs)
        idx = []
        for i, sg in enumerate(sigs):
            if sg is None:
                res[i] = OperationError("SignatureNotSet")
            elif len(sg.h) != 56 or len(sg.z) != 56 or (not prepared and len(pub_keys[i]) != 112):
                res[i] = OperationError("SignatureVerificationFailure")
            else:
                idx.append(i)
        h = b"".join(sigs[i].h for i in idx)
        z = b"".join(sigs[i].z for i in idx)
        pub = pub_keys if prepared else b"".join(pub_keys[i] for i in idx)
        return VerifyStream(self.engine.ed448_verify_stream(pub, h, z, int(d)), idx, res)

    # ---- messages fed twice in pieces -------------------------------------------------------------------
    def sign_stream(self, keys: Sequence[KeyPair] | Sequence[bytes], d: SecParam) -> "SignStream":
        """one sign() per key pair (or password) whose message is fed twice: update() in pass 1, next_pass(), the same
        bytes again through update(), then finish() -> a Signature per message, as sign() gives for the concatenated
        pieces, or OperationError("OperationResultNotSet") where pass 2 carried other bytes than pass 1.  D224 is refused
        (ValueError)."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("sign_stream: D224 is not resumable (quirk Q7)")
        pd, po = pack([k.priv_key if isinstance(k, KeyPair) else bytes(k) for k in keys])
        return SignStream(self.engine.ed448_sign_stream(pd, po, int(d)))

    def sha3_decrypt_stream(self, pws: Sequence[bytes], nonces: Sequence[bytes], tags: Sequence[bytes],
                            d: SecParam) -> "DecryptStream":
        """one sha3_decrypt per password whose ciphertext is fed twice: update() in pass 1 releases nothing, next_pass()
        gives the verdicts (None or SHA3DecryptionFailure), decrypt() takes the same bytes again and returns the plaintext
        pieces (the ciphertext for a failed message), finish() the final result, which also checks that both passes
        carried the same bytes.  All nonces have one length.  D224 is refused (ValueError)."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("sha3_decrypt_stream: D224 is not resumable (quirk Q7)")
        nl = len(nonces[0]) if nonces else 0
        if len(nonces) != len(pws) or len(tags) != len(pws) or any(len(z) != nl for z in nonces):
            raise ValueError("sha3_decrypt_stream: one nonce (all of one length) and one tag per password")
        pd, po = pack(pws)
        tb = b"".join(bytes(t).ljust(64, b"\0")[:64] for t in tags)
        st = self.engine.sponge_decrypt_stream(pd, po, b"".join(nonces), nl, tb, int(d))
        return DecryptStream(st, "SHA3DecryptionFailure", [len(t) != 64 for t in tags])

    def key_decrypt_stream(self, pws: Sequence[bytes], asym_nonces: Sequence[bytes], tags: Sequence[bytes],
                           d: SecParam) -> "DecryptStream":
        """as sha3_decrypt_stream for key_decrypt: asym_nonces are the Z of the messages (112 bytes each); failures are
        KeyDecryptionError, an off-curve Z included."""
        d = SecParam.try_from(int(d))
        if d == SecParam.D224:
            raise ValueError("key_decrypt_stream: D224 is not resumable (quirk Q7)")
        if len(asym_nonces) != len(pws) or len(tags) != len(pws) or any(len(z) != 112 for z in asym_nonces):
            raise ValueError("key_decrypt_stream: one 112-byte Z and one tag per password")
        pd, po = pack(pws)
        tb = b"".join(bytes(t).ljust(56, b"\0")[:56] for t in tags)
        st = self.engine.ed448_key_decrypt_stream(pd, po, b"".join(asym_nonces), tb, int(d))
        return DecryptStream(st, "KeyDecryptionError", [len(t) != 56 for t in tags])

    # ---- KeyPair::new ----------------------------------------------------------------------------------
    def new_keypairs(self, pws: Sequence[bytes], owner: str, d: SecParam) -> list[KeyPair]:
        d = SecParam.try_from(int(d))
        pd, po = pack(pws)
        pub = self.engine.ed448_keygen(pd, po, int(d))
        return [KeyPair(owner=owner, pub_key=row.tobytes(), priv_key=bytes(pw)) for pw, row in zip(pws, pub)]

    # ---- Signable ----------------------------------------------------------------------------------------
    def sign(self, msgs: Sequence[Message], keys: Sequence[KeyPair], d: SecParam) -> None:
        d = SecParam.try_from(int(d))
        pd, po = pack([k.priv_key for k in keys])
        md, mo = pack([m.msg for m in msgs])
        h, z = self.engine.ed448_sign(pd, po, md, mo, int(d))
        for m, hr, zr in zip(msgs, h, z):
            m.sig = Signature(h=hr.tobytes(), z=zr.tobytes())
            m.d = d

    def verify(self, msgs: Sequence[Message], pub_keys: Sequence[bytes]) -> list[Optional[OperationError]]:
        """Per message: None for Ok(()), else the OperationError the reference would return
        (SignatureNotSet / SecurityParameterNotSet / SignatureVerificationFailure, signable.rs:72-86)."""
        res: list[Optional[OperationError]] = [None] * len(msgs)
        groups: dict[int, list[int]] = {}
        for i, m in enumerate(msgs):
            if m.sig is None:
                res[i] = OperationError("SignatureNotSet")
            elif m.d is None:
                res[i] = OperationError("SecurityParameterNotSet")
            elif len(m.sig.h) != 56 or len(m.sig.z) != 56 or len(pub_keys[i]) != 112:
                # a malformed signature or key fails on its own and is left out of the fixed-stride batch (one short
                # field would otherwise shift every later item); the reference rejects it at the type level
                res[i] = OperationError("SignatureVerificationFailure")
            else:
                groups.setdefault(int(m.d), []).append(i)
        for d, idx in groups.items():
            md, mo = pack([msgs[i].msg for i in idx])
            pub = np.frombuffer(b"".join(pub_keys[i] for i in idx), dtype=np.uint8)
            h = np.frombuffer(b"".join(msgs[i].sig.h for i in idx), dtype=np.uint8)
            z = np.frombuffer(b"".join(msgs[i].sig.z for i in idx), dtype=np.uint8)
            _, ok = self.engine.ed448_verify(pub, md, mo, h, z, d)
            for i, o in zip(idx, ok):
                if not o:
                    res[i] = OperationError("SignatureVerificationFailure")
        return res

    # ---- one signer / one recipient --------------------------------------------------------------------
    def prepare_public_key(self, pub_key: bytes) -> PreparedPublicKey:
        """Prepares one public key (affine x || y, 112 bytes) for verify_prepared / key_encrypt_prepared: worth it when
        the key is used for many messages, over one call or several.  OperationError("InvalidPublicKey") when the point
        is not on the curve.  Close the key (or use it in a `with` block) before the engine."""
        if len(pub_key) != 112:
            raise OperationError("InvalidPublicKey")
        try:
            return self.engine.ed448_pub_prepare(pub_key)
        except CapyError as e:
            if e.status == ERR_BAD_POINT:
                raise OperationError("InvalidPublicKey") from None
            raise

    def verify_prepared(self, msgs: Sequence[Message], key: PreparedPublicKey) -> list[Optional[OperationError]]:
        """verify() with key as every message's public key: the same result per message."""
        res: list[Optional[OperationError]] = [None] * len(msgs)
        groups: dict[int, list[int]] = {}
        for i, m in enumerate(msgs):
            if m.sig is None:
                res[i] = OperationError("SignatureNotSet")
            elif m.d is None:
                res[i] = OperationError("SecurityParameterNotSet")
            elif len(m.sig.h) != 56 or len(m.sig.z) != 56:
                res[i] = OperationError("SignatureVerificationFailure")
            else:
                groups.setdefault(int(m.d), []).append(i)
        for d, idx in groups.items():
            md, mo = pack([msgs[i].msg for i in idx])
            h = np.frombuffer(b"".join(msgs[i].sig.h for i in idx), dtype=np.uint8)
            z = np.frombuffer(b"".join(msgs[i].sig.z for i in idx), dtype=np.uint8)
            ok = self.engine.ed448_verify_prepared(key, md, mo, h, z, d)
            for i, o in zip(idx, ok):
                if not o:
                    res[i] = OperationError("SignatureVerificationFailure")
        return res

    def key_encrypt_prepared(self, msgs: Sequence[Message], key: PreparedPublicKey, d: SecParam,
                             k_rand: Optional[Sequence[bytes]] = None) -> None:
        """key_encrypt() with key as every message's recipient: the same fields, the same bytes."""
        d = SecParam.try_from(int(d))
        if k_rand is None:
            k_rand = [os.urandom(56) for _ in msgs]
        if len(k_rand) != len(msgs) or any(len(k) != 56 for k in k_rand):
            raise ValueError("key_encrypt_prepared: one 56-byte nonce per message")
        md, mo = pack([m.msg for m in msgs])
        ct, tag, z = self.engine.ed448_key_encrypt_prepared(key, b"".join(k_rand), md, mo, int(d))
        for i, m in enumerate(msgs):
            m.msg = bytearray(ct[int(mo[i]):int(mo[i + 1])].tobytes())
            m.digest = tag[i].tobytes()
            m.asym_nonce = z[i].tobytes()
            m.d = d

    # ---- SpongeEncryptable ---------------------------------------------------------------------------
    def sha3_encrypt(self, msgs: Sequence[Message], pws: Sequence[bytes], d: SecParam,
                     nonces: Optional[Sequence[bytes]] = None) -> None:
        """Batched Message::sha3_encrypt (sha3/encryptable.rs:29-45): replaces .msg with the ciphertext, .digest with
        the tag, .sym_nonce with z, .d with d.  z = 512 random bytes per message (get_random_bytes(512), :31), drawn
        here on the host unless injected."""
        d = SecParam.try_from(int(d))
        if nonces is None:
            nonces = [os.urandom(512) for _ in msgs]
        if len(nonces) != len(msgs) or len(pws) != len(msgs) or any(len(z) != 512 for z in nonces):
            raise ValueError("sha3_encrypt: one password and one 512-byte nonce per message")
        pd, po = pack(pws)
        md, mo = pack([m.msg for m in msgs])
        ct, tag = self.engine.sponge_encrypt(pd, po, b"".join(nonces), 512, md, mo, int(d))
        for i, m in enumerate(msgs):
            m.msg = bytearray(ct[int(mo[i]):int(mo[i + 1])].tobytes())
            m.digest = tag[i].tobytes()
            m.sym_nonce = bytes(nonces[i])
            m.d = d

    def sha3_decrypt(self, msgs: Sequence[Message], pws: Sequence[bytes]) -> list[Optional[OperationError]]:
        """Batched Message::sha3_decrypt (:58-83).  Per message None for Ok(()), else SecurityParameterNotSet /
        SymNonceNotSet / SHA3DecryptionFailure; on failure .msg keeps the ciphertext."""
        res: list[Optional[OperationError]] = [None] * len(msgs)
        groups: dict[int, list[int]] = {}
        for i, m in enumerate(msgs):
            if m.d is None:
                res[i] = OperationError("SecurityParameterNotSet")
            elif m.sym_nonce is None:
                res[i] = OperationError("SymNonceNotSet")
            else:
                groups.setdefault((int(m.d), len(m.sym_nonce)), []).append(i)
        for (d, nl), idx in groups.items():
            pd, po = pack([pws[i] for i in idx])
            cd, co = pack([msgs[i].msg for i in idx])
            tags = b"".join(bytes(msgs[i].digest).ljust(64, b"\0")[:64] for i in idx)
            out, ok = self.engine.sponge_decrypt(pd, po, b"".join(msgs[i].sym_nonce for i in idx), nl, cd, co, tags, d)
            for j, i in enumerate(idx):
                good = bool(ok[j]) and len(msgs[i].digest) == 64
                if good:
                    msgs[i].msg = bytearray(out[int(co[j]):int(co[j + 1])].tobytes())
                else:
                    res[i] = OperationError("SHA3DecryptionFailure")
        return res

    # ---- KeyEncryptable ------------------------------------------------------------------------------
    def key_encrypt(self, msgs: Sequence[Message], pub_keys: Sequence[bytes], d: SecParam,
                    k_rand: Optional[Sequence[bytes]] = None) -> None:
        """Batched Message::key_encrypt (ecc/encryptable.rs:34-50): .msg <- ciphertext, .digest <- tag (56 bytes),
        .asym_nonce <- Z = [k]G (affine x || y), .d <- d.  k = 56 random bytes per message (:36) unless injected."""
        d = SecParam.try_from(int(d))
        if k_rand is None:
            k_rand = [os.urandom(56) for _ in msgs]
        if len(pub_keys) != len(msgs) or len(k_rand) != len(msgs):
            raise ValueError("key_encrypt: one public key and one nonce per message")
        for i in range(len(msgs)):
            if len(pub_keys[i]) != 112 or len(k_rand[i]) != 56:
                # (an ExtendedPoint / a 56-byte get_random_bytes in the reference: cannot be malformed there)
                raise ValueError(f"key_encrypt: item {i}: public key must be 112 bytes and the nonce 56 bytes")
        md, mo = pack([m.msg for m in msgs])
        rc, ct, tag, z = self.engine.ed448_key_encrypt(b"".join(pub_keys), b"".join(k_rand), md, mo, int(d))
        if rc:
            raise OperationError("InvalidPublicKey")
        for i, m in enumerate(msgs):
            m.msg = bytearray(ct[int(mo[i]):int(mo[i + 1])].tobytes())
            m.digest = tag[i].tobytes()
            m.asym_nonce = z[i].tobytes()
            m.d = d

    def key_decrypt(self, msgs: Sequence[Message], pws: Sequence[bytes]) -> list[Optional[OperationError]]:
        """Batched Message::key_decrypt (:72-94): None for Ok(()), else SymNonceNotSet (sic, :73) /
        SecurityParameterNotSet / KeyDecryptionError; on failure .msg keeps the ciphertext."""
        res: list[Optional[OperationError]] = [None] * len(msgs)
        groups: dict[int, list[int]] = {}
        for i, m in enumerate(msgs):
            if m.asym_nonce is None:
                res[i] = OperationError("SymNonceNotSet")
            elif m.d is None:
                res[i] = OperationError("SecurityParameterNotSet")
            elif len(m.asym_nonce) != 112:
                res[i] = OperationError("KeyDecryptionError")  # not a point encoding: fails alone, stays out of the batch
            else:
                groups.setdefault(int(m.d), []).append(i)
        for d, idx in groups.items():
            pd, po = pack([pws[i] for i in idx])
            cd, co = pack([msgs[i].msg for i in idx])
            tags = b"".join(bytes(msgs[i].digest).ljust(56, b"\0")[:56] for i in idx)
            _, out, ok = self.engine.ed448_key_decrypt(pd, po, b"".join(msgs[i].asym_nonce for i in idx), cd, co, tags, d)
            for j, i in enumerate(idx):
                good = bool(ok[j]) and len(msgs[i].digest) == 56
                if good:
                    msgs[i].msg = bytearray(out[int(co[j]):int(co[j + 1])].tobytes())
                else:
                    res[i] = OperationError("KeyDecryptionError")
        return res


class SpongeStream:
    """Streams of Gpu.sha3_stream / Gpu.kmac_xof_stream: update() appends one piece per stream, finish() ends them.
    Use it in a `with` block (or call close()) to release its device memory before the engine."""

    def __init__(self, hasher: Hasher, d: int):
        self.hasher = hasher
        self.d = d

    def update(self, pieces: Sequence[bytes]) -> None:
        data, off = pack(pieces)
        self.hasher.update(data, off)

    def finish(self, l: Optional[int] = None) -> list[bytes]:
        """SHA3-d: the digests (l must be None or d).  KMACXOF: l output bits per stream (default d)."""
        out = self.hasher.final(self.d if l is None else l)
        return [r.tobytes() for r in out]

    def close(self) -> None:
        self.hasher.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class EncryptStream:
    """Streams of Gpu.sha3_encrypt_stream / Gpu.key_encrypt_stream: update() encrypts one piece per message, finish()
    returns the tags.  Use it in a `with` block (or call close()) to release its device memory before the engine."""

    def __init__(self, stream, nonces: Optional[list[bytes]] = None, asym_nonces: Optional[list[bytes]] = None):
        self.stream = stream
        self.nonces = nonces
        self.asym_nonces = asym_nonces

    def update(self, pieces: Sequence[bytes]) -> list[bytes]:
        data, off = pack(pieces)
        ct = self.stream.update(data, off)
        return [ct[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(pieces))]

    def finish(self) -> list[bytes]:
        return [r.tobytes() for r in self.stream.final()]

    def close(self) -> None:
        self.stream.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class VerifyStream:
    """Streams of Gpu.verify_stream: update() appends one piece per message (all of them, the failed ones included),
    finish() gives verify()'s result per message."""

    def __init__(self, stream, idx: list[int], res: list[Optional[OperationError]]):
        self.stream = stream
        self.idx = idx
        self.res = res

    def update(self, pieces: Sequence[bytes]) -> None:
        if len(pieces) != len(self.res):
            raise ValueError(f"verify_stream update: {len(pieces)} pieces for {len(self.res)} messages")
        data, off = pack([pieces[i] for i in self.idx])
        self.stream.update(data, off)

    def finish(self) -> list[Optional[OperationError]]:
        _, ok = self.stream.final()
        for i, o in zip(self.idx, ok):
            if not o:
                self.res[i] = OperationError("SignatureVerificationFailure")
        return self.res

    def close(self) -> None:
        self.stream.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class SignStream:
    """Streams of Gpu.sign_stream: update() one piece per message in each pass, next_pass() between the passes,
    finish() the signatures."""

    def __init__(self, stream):
        self.stream = stream

    def update(self, pieces: Sequence[bytes]) -> None:
        self.stream.update(*pack(pieces))

    def next_pass(self) -> None:
        self.stream.next_pass()

    def finish(self) -> list[Signature | OperationError]:
        h, z, ok = self.stream.final()
        return [Signature(h=hr.tobytes(), z=zr.tobytes()) if o else OperationError("OperationResultNotSet")
                for hr, zr, o in zip(h, z, ok)]

    def close(self) -> None:
        self.stream.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class DecryptStream:
    """Streams of Gpu.sha3_decrypt_stream / Gpu.key_decrypt_stream: update() the ciphertext pieces of pass 1,
    next_pass() -> verdicts, decrypt() the same pieces again -> plaintext pieces, finish() -> the results."""

    def __init__(self, stream, error: str, bad_tag: list[bool]):
        self.stream = stream
        self.error = error
        self.bad_tag = bad_tag  # a tag of the wrong length fails, as in the one-shot calls

    def _results(self, ok) -> list[Optional[OperationError]]:
        return [None if o and not b else OperationError(self.error) for o, b in zip(ok, self.bad_tag)]

    def update(self, pieces: Sequence[bytes]) -> None:
        self.stream.update(*pack(pieces))

    def next_pass(self) -> list[Optional[OperationError]]:
        return self._results(self.stream.next_pass()[1])

    def decrypt(self, pieces: Sequence[bytes]) -> list[bytes]:
        data, off = pack(pieces)
        out = self.stream.decrypt(data, off)
        return [out[int(off[i]):int(off[i + 1])].tobytes() for i in range(len(pieces))]

    def finish(self) -> list[Optional[OperationError]]:
        return self._results(self.stream.final()[1])

    def close(self) -> None:
        self.stream.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _append_reference_padding(msg: bytearray, d: int) -> None:
    """What shake() leaves behind in Message.msg (shake_functions.rs:24-29 + sponge.rs:13-15,89-95)."""
    msg.append(0x86 if len(msg) % 136 == 135 else 0x06)
    c = {224: 448, 256: 512, 384: 768, 512: 1024}[d]
    r = (1600 - c) // 8
    if len(msg) % r:
        q = r - len(msg) % r
        msg.extend(bytes(q - 1) + b"\x80")
