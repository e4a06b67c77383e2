"""CPU suite for prepared public keys: the comb code of capycrypt_b200/csrc/ed448.cuh that the CUDA kernels run, compiled
for the CPU by tests/host/ed448_prepared_host_check.cpp (built here) and checked against the oracle.

  - the window builder given G reproduces G's table bit for bit;
  - V's table built from the affine multiples (j+1) * 32^i * V, as fb_table_kernel builds it, equals the window builder's;
  - a comb over V's table gives [h]V and the joint comb gives [z]G + [h]V, with h and z unreduced (quirk Q10)."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import ref_ed448 as E

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host", "ed448_prepared_host_check.cpp")
P, R = E.P, E.R


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("prepared") / "libed448_prepared_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", lib, SRC], check=True)
    h = C.CDLL(lib)
    h.host_table_words.restype = C.c_size_t
    return h


def _table(host, fn, *args):
    t = np.zeros(host.host_table_words(), dtype=np.uint32)
    fn(*args, t.ctypes.data)
    return t


def _multiples(pt):
    """(j+1) * 32^i * pt for i < 90, j < 16 as affine bytes, item 16 i + j"""
    out, base = [], pt
    for i in range(90):
        acc = base
        for j in range(16):
            out.append(E.point_to_bytes(acc))
            acc = E.point_add(acc, base)
        for _ in range(5):
            base = E.point_add(base, base)
    return b"".join(out)


@pytest.fixture(scope="module")
def table_g(host):
    return _table(host, host.host_table_g)


@pytest.fixture(scope="module")
def v_and_table(host):
    v = E.scalar_mult(random.Random(11).randrange(1, R), E.GENERATOR)
    return v, _table(host, host.host_table_of, E.point_to_bytes(v))


def test_window_builder_given_g_reproduces_g_table(host, table_g):
    t = _table(host, host.host_table_of, E.point_to_bytes(E.GENERATOR))
    assert np.array_equal(t, table_g)


@pytest.mark.parametrize("which", ["G", "V", "identity"])
def test_table_from_affine_multiples_equals_window_builder(host, table_g, v_and_table, which):
    pt, want = {"G": (E.GENERATOR, table_g), "V": v_and_table,
                "identity": (E.IDENTITY, _table(host, host.host_table_of, E.point_to_bytes(E.IDENTITY)))}[which]
    got = _table(host, host.host_table_from_points, _multiples(pt))
    assert np.array_equal(got, want)


def test_identity_table_is_all_neutral_entries(host):
    t = _table(host, host.host_table_of, E.point_to_bytes(E.IDENTITY)).reshape(-1, 48)
    assert (t[:, 0] == 1).all() and (t[:, 16] == 1).all()
    assert not t[:, 1:16].any() and not t[:, 17:].any()


SCALARS = [0, 1, 2, 15, 16, 17, R - 1, R, R + 1, 2 * R + 5, 2**446 - 1, 2**448 - 1, int("8" * 112, 16),
           int("f" * 112, 16)]


def test_comb_over_v_table(host, v_and_table):
    v, tv = v_and_table
    rnd = random.Random(12)
    out = (C.c_uint8 * 112)()
    for k in SCALARS + [rnd.randrange(2**448) for _ in range(8)]:
        for ct in (0, 1):
            host.host_comb(k.to_bytes(56, "big"), tv.ctypes.data, ct, out)
            assert bytes(out) == E.point_to_bytes(E.scalar_mult(k, v)), (k, ct)


def test_joint_comb_is_zg_plus_hv(host, table_g, v_and_table):
    v, tv = v_and_table
    rnd = random.Random(13)
    out = (C.c_uint8 * 112)()
    pairs = [(0, 0), (0, 1), (1, 0), (R, R), (R - 1, R + 1), (2**448 - 1, 2**448 - 1)]
    pairs += [(rnd.choice(SCALARS), rnd.randrange(2**448)) for _ in range(4)]
    pairs += [(rnd.randrange(2**448), rnd.randrange(2**448)) for _ in range(6)]
    for z, h in pairs:
        for ct in (0, 1):
            host.host_joint_comb(z.to_bytes(56, "big"), h.to_bytes(56, "big"), table_g.ctypes.data, tv.ctypes.data, ct, out)
            want = E.point_add(E.scalar_mult(z, E.GENERATOR), E.scalar_mult(h, v))
            assert bytes(out) == E.point_to_bytes(want), (z, h, ct)


def test_joint_comb_with_v_equal_g_and_identity(host, table_g):
    out = (C.c_uint8 * 112)()
    t_id = _table(host, host.host_table_of, E.point_to_bytes(E.IDENTITY))
    z, h = 2**447 + 12345, 2**440 + 99
    host.host_joint_comb(z.to_bytes(56, "big"), h.to_bytes(56, "big"), table_g.ctypes.data, table_g.ctypes.data, 1, out)
    assert bytes(out) == E.point_to_bytes(E.scalar_mult(z + h, E.GENERATOR))
    host.host_joint_comb(z.to_bytes(56, "big"), h.to_bytes(56, "big"), table_g.ctypes.data, t_id.ctypes.data, 0, out)
    assert bytes(out) == E.point_to_bytes(E.scalar_mult(z, E.GENERATOR))
