"""CPU: the header of a hasher blob (capy_hasher_blob_info, include/capy_gpu.h).  Hand-built headers of every kind and d
are accepted with the lengths they declare, and each malformed one is refused.  The library loads without a GPU."""
from __future__ import annotations

import ctypes as C
import struct

import numpy as np
import pytest

from capycrypt_b200 import _binding as B
from capycrypt_b200.engine import hasher_blob_info

SHA3_RATE = {224: 144, 256: 136, 384: 104, 512: 72}
KMAC_RATE = {256: 168, 384: 152, 512: 136}
VALID = [(0, d, r) for d, r in SHA3_RATE.items()] + [(1, d, r) for d, r in KMAC_RATE.items()]


@pytest.fixture(scope="module")
def lib():
    return B.load()


def header(kind, d, rate, n, *, magic=b"CAPYHSTR", version=1, rec=None, zero=0, pad=b"\0" * 24):
    rec = 208 + rate if rec is None else rec
    return magic + struct.pack("<IIIIIIQ", version, kind, d, rate, rec, zero, n) + pad


def blob(kind, d, rate, n, **kw):
    return header(kind, d, rate, n, **kw) + bytes(n * (208 + rate))


def info(lib, b: bytes, length=None):
    a = np.frombuffer(b, np.uint8) if b else np.zeros(1, np.uint8)
    kind, d, n = C.c_int(-1), C.c_int(-1), C.c_uint64(7)
    rc = lib.capy_hasher_blob_info(a.ctypes.data, len(b) if length is None else length, C.byref(kind), C.byref(d),
                                   C.byref(n))
    return rc, (kind.value, d.value, n.value)


@pytest.mark.parametrize("kind,d,rate", VALID)
@pytest.mark.parametrize("n", [0, 1, 3])
def test_valid_headers(lib, kind, d, rate, n):
    assert (208 + rate) % 8 == 0
    rc, got = info(lib, blob(kind, d, rate, n))
    assert rc == B.OK and got == (kind, d, n)
    assert hasher_blob_info(blob(kind, d, rate, n), lib) == (kind, d, n)


def test_null_outputs_and_null_blob(lib):
    b = np.frombuffer(blob(0, 256, 136, 2), np.uint8)
    assert lib.capy_hasher_blob_info(b.ctypes.data, b.size, None, None, None) == B.OK
    assert lib.capy_hasher_blob_info(None, 64, None, None, None) == B.ERR_BAD_ARG


MALFORMED = {
    "magic": lambda: blob(0, 256, 136, 1, magic=b"CAPYHSTX"),
    "version 0": lambda: blob(0, 256, 136, 1, version=0),
    "version 2": lambda: blob(0, 256, 136, 1, version=2),
    "kind 2": lambda: blob(2, 256, 136, 1),
    "kind of another rate": lambda: blob(1, 256, 136, 1),
    "d 300": lambda: blob(0, 300, 136, 1),
    "d 0": lambda: blob(0, 0, 136, 1),
    "kmac d224": lambda: blob(1, 224, 172, 1),
    "kmac d224 at 168": lambda: blob(1, 224, 168, 1),
    "rate": lambda: blob(0, 256, 144, 1),
    "record": lambda: header(0, 256, 136, 1, rec=208 + 136 + 8) + bytes(352),
    "record 0": lambda: header(0, 256, 136, 0, rec=0),
    "zero field": lambda: blob(0, 256, 136, 1, zero=1),
    "reserved byte": lambda: blob(0, 256, 136, 1, pad=b"\0" * 23 + b"\1"),
    "one byte short": lambda: blob(0, 256, 136, 2)[:-1],
    "one byte long": lambda: blob(0, 256, 136, 2) + b"\0",
    "a record short": lambda: blob(0, 256, 136, 2)[:-344],
    "n huge": lambda: header(0, 256, 136, (1 << 64) - 1) + bytes(344),
    "n overflows": lambda: header(1, 512, 136, (1 << 64) // 344 + 1) + bytes(344),
    "header short": lambda: blob(0, 256, 136, 0)[:63],
    "empty": lambda: b"",
}


@pytest.mark.parametrize("case", sorted(MALFORMED))
def test_malformed_headers(lib, case):
    rc, got = info(lib, MALFORMED[case]())
    assert rc == B.ERR_BAD_ARG, case
    assert got == (-1, -1, 7), "outputs are left alone on an error"
    with pytest.raises(B.CapyError) as e:
        hasher_blob_info(MALFORMED[case](), lib)
    assert e.value.status == B.ERR_BAD_ARG


def test_length_argument_is_what_counts(lib):
    b = blob(0, 512, 72, 3)
    assert info(lib, b, len(b) - 280)[0] == B.ERR_BAD_ARG  # the buffer holds more than the length says
    assert info(lib, b + bytes(280), len(b))[0] == B.OK
