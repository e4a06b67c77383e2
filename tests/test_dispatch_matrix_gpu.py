"""GPU: every kernel the launchers can choose, each checked bit-exactly against the oracle.

The other GPU tests are organised by operation; this file is organised by launch path.  Each case calls a `_dev` entry
point at a shape chosen to land in one kernel instantiation and mode (plain, throttled, tiered, chain-cut, dependent
jobs, split last row, ...), reads what actually launched from a torch.profiler trace, and compares the result with the
oracle -- the whole batch, or for large batches a seeded sample that always holds item 0, the last item and the items of
the last partial 128-item block.  Where a switch exists (CAPY_NO_CHAIN_SPLIT, CAPY_FLAG_NO_SORT, CAPY_FLAG_NO_PAIR, the
forced warp-sharing classes) the switched twin must give the same bytes.

Every device output and byte input is carved out of a larger buffer with 4 KiB of a seeded pattern on each side, at
offset 0 or at an odd offset: a kernel that writes past its output, or stores at the wrong address, changes a guard byte.
Offset arrays stay 8-byte aligned (uint64 in the ABI).

The last test checks that the cases together launched every kernel of the library (KERNELS); tests/test_kernel_list.py
checks KERNELS against the kernels compiled into libcapycrypt_gpu.so.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import re

import numpy as np
import pytest

from capycrypt_b200.engine import pack
from oracle import ref_ed448 as E
from oracle import ref_sha3 as R

pytestmark = pytest.mark.gpu

LANES = (9, 13, 17, 18, 19, 21)
KERNELS = frozenset(
    ["ae_concat_kernel", "ae_finish_kernel", "any_bad_kernel", "fb_table_kernel", "fixed_base_kernel",
     "len_hist_kernel", "len_scan_kernel", "len_scatter_kernel", "scalar_prep_kernel", "sign_finish_kernel",
     "var_base_kernel", "verify_compare_kernel", "to_affine_kernel<16>"]
    + [f"prefix_state_kernel<{L}>" for L in (17, 19, 21)]
    + [f"sha3_short_kernel<17,{m}>" for m in (2, 4, 6, 8, 10, 12, 14, 16)]
    + [f"sha3_short_kernel<9,{m}>" for m in (2, 4, 6, 8)]
    + [f"sha3_uniform_kernel<{L}>" for L in (9, 13, 17, 18)]
    + [f"{k}<{L}>" for k in ("sponge_kernel", "sponge_tiered_kernel", "sponge_chain_kernel") for L in LANES]
    + [f"sponge_kernel2<{L}>" for L in (17, 19, 21)]
)
assert len(KERNELS) == 53

NO_SORT, NO_PAIR, COSCHED_SHIFT = 1, 2, 8
SHA3_LANES = {224: 18, 256: 17, 384: 13, 512: 9}  # rate / 8 of SHA3-d
KMAC_LANES = {224: 21, 256: 21, 384: 19, 512: 17}  # whole lanes of the cSHAKE / KMAC rate (172 bytes at D224)
SHA3_RATE = {224: 144, 256: 136, 384: 104, 512: 72}
KMAC_RATE = {224: 172, 256: 168, 384: 152, 512: 136}
GUARD = 4096


def normalise_kernel(name: str) -> str:
    """'void capy::sha3_short_kernel<(int)17, (int)2>(const uint4 *, ...)' -> 'sha3_short_kernel<17,2>'"""
    s = name.strip()
    if s.startswith("void "):
        s = s[5:]
    s = s.replace("capy::", "")
    s = re.sub(r"\((?:unsigned )?int\)", "", s)
    s = s.split("(", 1)[0]
    return s.replace(" ", "")


# ---- bookkeeping of the coverage test -------------------------------------------------------------------------------
SEEN: set[str] = set()
PASSED: set[str] = set()
CASES: dict = {}


def case(fn):
    CASES[fn.__name__] = fn
    return fn


# ---- launches ----------------------------------------------------------------------------------------------------------
class Launch:
    def __init__(self, e):
        a = e.get("args", {})
        self.raw = e["name"]
        self.name = normalise_kernel(e["name"])
        self.grid = tuple(a.get("grid", ()))
        self.block = tuple(a.get("block", ()))
        self.smem = a.get("shared memory")

    def __repr__(self):
        return f"{self.name} grid={self.grid} block={self.block} smem={self.smem}"


class Ctx:
    def __init__(self, eng, orc, tmp_path, monkeypatch):
        import torch

        self.torch = torch
        self.eng = eng
        self.orc = orc
        self.tmp = tmp_path
        self.mp = monkeypatch
        self.sm = torch.cuda.get_device_properties(0).multi_processor_count
        self.traces = 0

    @property
    def stream(self):
        return C.c_void_p(self.torch.cuda.current_stream().cuda_stream)

    def launched(self, fn, eng=None):
        """Runs fn under torch.profiler (CUDA activities) and returns the capy:: kernels it launched, in order."""
        from torch.profiler import ProfilerActivity, profile

        torch = self.torch
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        self.traces += 1
        path = self.tmp / f"trace{self.traces}.json"
        prof.export_chrome_trace(str(path))
        with open(path) as f:
            events = json.load(f)["traceEvents"]
        ks = [Launch(e) for e in events if e.get("cat") == "kernel" and "capy::" in e.get("name", "")]
        assert ks, "no capy:: kernel in the profiler trace"
        SEEN.update(k.name for k in ks)
        return ks

    def call(self, fname, *args, eng=None):
        eng = eng or self.eng
        rc = getattr(eng.lib, fname)(eng._ctx, 0, self.stream, *args)
        return eng._check(rc, allow=(-4,))


def names(ks):
    return [k.name for k in ks]


def only(ks, name):
    got = [k for k in ks if k.name == name]
    assert got, f"expected {name}, launched {ks}"
    return got


def absent(ks, name):
    assert not [k for k in ks if k.name == name], f"{name} must not launch here: {ks}"


# ---- guarded device buffers ----------------------------------------------------------------------------------------------
class Guarded:
    """`nbytes` of device memory at `offset` inside a buffer with GUARD bytes of a seeded pattern on each side"""

    def __init__(self, ctx, nbytes, offset=0, fill=None, seed=0):
        torch = ctx.torch
        self.lo = GUARD + offset
        self.hi = self.lo + nbytes
        rnd = np.random.default_rng(10_000 + seed + 7 * offset + nbytes % 9973)
        host = rnd.integers(0, 256, size=self.hi + GUARD, dtype=np.uint8)
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
        bad = np.nonzero(whole[self.hi:] != self.pattern[self.hi:])[0]
        assert bad.size == 0, f"write past the end of the buffer: guard bytes {bad[:8]} changed"
        return whole[self.lo:self.hi].copy()


def dev_off(ctx, off):
    return ctx.torch.from_numpy(np.ascontiguousarray(off, dtype=np.int64)).cuda()


def ragged(rnd, lens):
    off = np.zeros(len(lens) + 1, np.uint64)
    off[1:] = np.cumsum(np.asarray(lens, dtype=np.uint64))
    return rnd.integers(0, 256, size=int(off[-1]), dtype=np.uint8), off


def sample(n, seed=0, k=600):
    """all items of a small batch; for a large one item 0, the last item, the last partial block and a seeded sample"""
    if n <= 4096:
        return np.arange(n)
    rnd = np.random.default_rng(seed)
    idx = set(rnd.choice(n, size=k, replace=False).tolist()) | {0, n - 1} | set(range(128 * ((n - 1) // 128), n))
    return np.array(sorted(idx))


def sub(data, off, idx):
    return pack([data[int(off[i]):int(off[i + 1])] for i in idx])


def rows(data, length, stride, idx):
    return pack([data[i * stride:i * stride + length] for i in idx])


def mismatch(got, want):
    bad = np.nonzero((got != want).reshape(len(got), -1).any(axis=1))[0]
    return f"{bad.size} items differ, first {bad[:10]}"


# ---- C ABI calls (raw pointers: the guarded buffers are views at odd addresses) ---------------------------------------------
def sha3_dev(ctx, d, data_g, off_t, n, out_g, flags=0):
    ctx.call("capy_sha3_batch_dev", d, data_g.ptr, off_t.data_ptr(), n, out_g.ptr, flags)


def sha3_fixed_dev(ctx, d, data_g, msg_len, stride, n, out_g):
    ctx.call("capy_sha3_batch_fixed_dev", d, data_g.ptr, msg_len, stride, n, out_g.ptr, 0)


def cshake_dev(ctx, d, data_g, off_t, n, fn, cs, out_bits, out_g, eng=None):
    f = np.frombuffer(fn or b"\0", np.uint8)
    s = np.frombuffer(cs or b"\0", np.uint8)
    ctx.call("capy_cshake_batch_dev", d, data_g.ptr, off_t.data_ptr(), n, f.ctypes.data, len(fn), s.ctypes.data, len(cs),
             out_bits, out_g.ptr, eng=eng)


def kmac_dev(ctx, d, keys_g, koff_t, data_g, off_t, n, cs, out_bits, out_g, out_off_t=None):
    s = np.frombuffer(cs or b"\0", np.uint8)
    ctx.call("capy_kmac_xof_batch_dev", d, keys_g.ptr, koff_t.data_ptr(), data_g.ptr, off_t.data_ptr(), n, s.ctypes.data,
             len(cs), out_bits, out_off_t.data_ptr() if out_off_t is not None else None, out_g.ptr)


def sha3_oracle(ctx, data, off, d, idx):
    sd, so = sub(data, off, idx)
    return ctx.orc.sha3_batch(sd, so, d, threads=0)


# =========================================================================================================================
# SHA3-d, fixed length (capy_sha3_batch_fixed_dev)
# =========================================================================================================================
def fixed_case(ctx, d, msg_len, stride, n, out_offset=0, data_offset=0, seed=0):
    rnd = np.random.default_rng(seed)
    total = (n - 1) * stride + msg_len  # the last row ends with its last message byte
    data = rnd.integers(0, 256, size=total, dtype=np.uint8)
    data_g = Guarded(ctx, total, data_offset, data, seed=1)
    out_g = Guarded(ctx, n * d // 8, out_offset, seed=2)
    ks = ctx.launched(lambda: sha3_fixed_dev(ctx, d, data_g, msg_len, stride, n, out_g))
    got = out_g.get().reshape(n, d // 8)
    idx = sample(n, seed)
    want = ctx.orc.sha3_batch(*rows(data, msg_len, stride, idx), d, threads=0)
    assert np.array_equal(got[idx], want), (d, msg_len, stride, n, mismatch(got[idx], want))
    return ks, got


@case
def sha3_short_d256(ctx):
    for m in (2, 4, 6, 8, 10, 12, 14, 16):
        ks, _ = fixed_case(ctx, 256, 8 * m, 8 * m, 1000 + m, seed=m)
        assert names(ks) == [f"sha3_short_kernel<17,{m}>"], ks


@case
def sha3_short_d512(ctx):
    for m in (2, 4, 6, 8):
        ks, _ = fixed_case(ctx, 512, 8 * m, 8 * m + 16, 999 + m, seed=m)
        assert names(ks) == [f"sha3_short_kernel<9,{m}>"], ks


@case
def sha3_short_shape_at_odd_output(ctx):
    """the single-block kernel stores 16-byte rows: an odd output address sends the batch to the byte-granular sponge"""
    for d in (256, 512):
        ks, _ = fixed_case(ctx, d, 64, 64, 700, out_offset=1, seed=d)
        assert names(ks) == [f"sponge_kernel<{SHA3_LANES[d]}>"], ks
        ks, _ = fixed_case(ctx, d, 64, 64, 700, data_offset=8, seed=d)  # 8- but not 16-byte aligned rows
        assert names(ks) == [f"sha3_uniform_kernel<{SHA3_LANES[d]}>"], ks


@case
def sha3_uniform_all_d(ctx):
    for d in (224, 256, 384, 512):
        ks, _ = fixed_case(ctx, d, 200, 208, 777, seed=d)
        assert names(ks) == [f"sha3_uniform_kernel<{SHA3_LANES[d]}>"], ks
        # 4-byte aligned output: the 4-byte granule stores
        ks, _ = fixed_case(ctx, d, 136, 136, 513, out_offset=4, seed=d + 1)
        assert names(ks) == [f"sha3_uniform_kernel<{SHA3_LANES[d]}>"], ks


@case
def sha3_fixed_last_row_split(ctx):
    """msg_len % 8 != 0 on a caller-owned buffer: n - 1 rows in the uniform kernel, the last row in the byte-granular
    sponge kernel, whose digest goes to out + (n - 1) * d / 8"""
    for d in (224, 256, 384, 512):
        for n in (2, 333):
            ks, _ = fixed_case(ctx, d, 101, 104, n, seed=d + n)
            L = SHA3_LANES[d]
            assert names(ks) == [f"sha3_uniform_kernel<{L}>", f"sponge_kernel<{L}>"], ks
            assert ks[1].grid == (1, 1, 1), ks
    # an odd output keeps every row in the sponge kernel
    ks, _ = fixed_case(ctx, 256, 101, 104, 333, out_offset=3, seed=5)
    assert names(ks) == ["sponge_kernel<17>"], ks


# =========================================================================================================================
# SHA3-d, ragged (capy_sha3_batch_dev): plain, throttled, tiered
# =========================================================================================================================
def ragged_sha3(ctx, d, data, off, flags=0, out_offset=1, data_offset=1, seed=0):
    n = len(off) - 1
    data_g = Guarded(ctx, len(data), data_offset, data, seed=seed)
    off_t = dev_off(ctx, off)
    out_g = Guarded(ctx, n * d // 8, out_offset, seed=seed + 1)
    ks = ctx.launched(lambda: sha3_dev(ctx, d, data_g, off_t, n, out_g, flags))
    return ks, out_g.get().reshape(n, d // 8)


def throttle_smem(w):
    return 227 * 1024 // w - 1024


def assert_throttled(k, w):
    assert k.block == (128, 1, 1) and k.smem is not None and 0 <= k.smem - throttle_smem(w) < 1024, (w, k)


@case
def sha3_ragged_small(ctx):
    """a small ragged batch is ordered on the device (histogram, scan, scatter) and runs throttled to W = 1"""
    for d in (224, 256, 384, 512):
        rnd = np.random.default_rng(d)
        data, off = ragged(rnd, rnd.integers(0, 700, size=1500))
        want = ctx.orc.sha3_batch(data, off, d, threads=0)
        L = SHA3_LANES[d]
        ks, got = ragged_sha3(ctx, d, data, off, seed=d)
        assert names(ks) == ["len_hist_kernel", "len_scan_kernel", "len_scatter_kernel", f"sponge_kernel<{L}>"], ks
        assert_throttled(ks[-1], 1)
        assert np.array_equal(got, want), mismatch(got, want)
        ks, got = ragged_sha3(ctx, d, data, off, flags=NO_SORT, seed=d)
        assert names(ks) == [f"sponge_kernel<{L}>"], ks
        assert ks[0].smem in (0, None) or ks[0].smem < 1024, ks
        assert np.array_equal(got, want), mismatch(got, want)


def expected_w(sm, blocks):
    """plan_from_hist's occupancy throttle for a batch of these per-item block counts (bin + 1)"""
    m = int(blocks.max())
    ideal = float(blocks.sum()) / (32.0 * 4.0 * sm)
    w = 0
    if m * 4.0 > 0.7 * ideal:
        w = 3
        if m * 3.0 > 0.7 * ideal:
            w = 2
        if m * 2.0 > 0.7 * ideal:
            w = 1
    return w


@case
def sha3_ragged_throttle_w2_w3(ctx):
    """batches whose longest item is short against the work: W = 2 or 3 one-warp blocks per scheduler"""
    d = 256
    rate = SHA3_RATE[d]
    for w, ratio in ((2, 3.6), (3, 5.0)):
        n = int(ratio / 0.75 * 128 * ctx.sm) // 2 * 2
        i = np.arange(n)
        lens = (i % 2) * rate + (i * 7) % rate  # bins 0 and 1 alternate: 1.5 blocks per item, 2 at most
        assert expected_w(ctx.sm, lens // rate + 1) == w
        rnd = np.random.default_rng(w)
        data, off = ragged(rnd, lens)
        ks, got = ragged_sha3(ctx, d, data, off, seed=w)
        assert names(ks) == ["len_hist_kernel", "len_scan_kernel", "len_scatter_kernel", "sponge_kernel<17>"], ks
        assert_throttled(ks[-1], w)
        idx = sample(n, w)
        want = sha3_oracle(ctx, data, off, d, idx)
        assert np.array_equal(got[idx], want), mismatch(got[idx], want)
        ks, got2 = ragged_sha3(ctx, d, data, off, flags=NO_SORT, seed=w)
        assert names(ks) == ["sponge_kernel<17>"], ks
        assert np.array_equal(got, got2)


def chain_bound(rnd, rate, short=3000):
    """a few long messages (block-boundary and quirk lengths included) among many short ones"""
    long_lens = [200_000, 150_001, 120_003, rate * 1500, rate * 1500 - 1, rate * 1500 + 1, 136 * 900 + 135,
                 rate * 1200 + rate - 1, 90_007, 90_006, 90_005, 90_004]
    lens = np.concatenate([long_lens, rnd.integers(0, 400, size=short)]).astype(np.int64)
    rnd.shuffle(lens)
    return lens


def tier_plan(ctx, lens, unit):
    """capy_plan_tiers3 on the length histogram of a batch: ([warp items with 1, 2, 3 chains per scheduler], pair items)"""
    bins = np.minimum(np.asarray(lens) // unit, 16383)
    cnt = np.bincount(bins, minlength=16384)
    cum = (cnt[::-1].cumsum()[::-1] - cnt).astype(np.uint32)  # items in bins > k
    w, p = np.zeros(3, np.uint64), np.zeros(1, np.uint64)
    ctx.eng._check(ctx.eng.lib.capy_plan_tiers3(cum.ctypes.data, len(cum), len(bins), int(bins.max()) + 1,
                                                int((bins + 1).sum()), ctx.sm, w.ctypes.data, p.ctypes.data))
    return w.tolist(), int(p[0])


@case
def sha3_tiered_and_twins(ctx):
    """chain-bound batches run tiered (384-thread blocks); NO_PAIR, NO_SORT and the forced warp-sharing classes give the
    same bytes"""
    for d in (224, 256, 384, 512):
        rnd = np.random.default_rng(40 + d)
        lens = chain_bound(rnd, SHA3_RATE[d])
        warp, pair = tier_plan(ctx, lens, SHA3_RATE[d])
        assert sum(warp) > 0 and pair > 0, (warp, pair)  # all three tiers, the pair tier storing at odd addresses
        data, off = ragged(rnd, lens)
        want = ctx.orc.sha3_batch(data, off, d, threads=0)
        L = SHA3_LANES[d]
        ks, got = ragged_sha3(ctx, d, data, off, seed=d)
        assert only(ks, f"sponge_tiered_kernel<{L}>")[0].block == (384, 1, 1), ks
        absent(ks, f"sponge_kernel<{L}>")
        assert np.array_equal(got, want), (d, mismatch(got, want))
        twins = [(NO_PAIR, f"sponge_kernel<{L}>"), (NO_SORT, f"sponge_kernel<{L}>")]
        if d == 256:
            twins += [(c << COSCHED_SHIFT, f"sponge_tiered_kernel<{L}>") for c in (1, 2, 3)]
        for flags, kern in twins:
            ks, got = ragged_sha3(ctx, d, data, off, flags=flags, seed=d + flags)
            assert names(ks)[-1] == kern, (flags, ks)
            if flags == NO_PAIR:
                assert_throttled(ks[-1], 1)
                absent(ks, f"sponge_tiered_kernel<{L}>")
            assert np.array_equal(got, want), (d, flags, mismatch(got, want))


# =========================================================================================================================
# chains cut in two (sponge_chain_kernel): uniform batches that fill the schedulers unevenly
# =========================================================================================================================
def chain_n(ctx):
    """2^16 + 37 items: uneven fill (3.46 warps per scheduler on 148 SMs) and a partial last block"""
    return (1 << 16) + 37


def assert_chain(ks, L, n):
    k = only(ks, f"sponge_chain_kernel<{L}>")[0]
    assert k.block == (128, 1, 1) and k.grid == (2 * ((n + 127) // 128), 1, 1), k


@case
def sha3_fixed_chain_cut(ctx):
    n = chain_n(ctx)
    for d in (224, 256, 384, 512):
        L = SHA3_LANES[d]
        msg_len = 12 * SHA3_RATE[d] + 8
        ks, got = fixed_case(ctx, d, msg_len, msg_len, n, out_offset=1 if d == 384 else 0, seed=d)
        assert names(ks) == [f"sponge_chain_kernel<{L}>"], ks
        assert_chain(ks, L, n)
        ctx.mp.setenv("CAPY_NO_CHAIN_SPLIT", "1")
        ks, got2 = fixed_case(ctx, d, msg_len, msg_len, n, seed=d)
        ctx.mp.delenv("CAPY_NO_CHAIN_SPLIT")
        assert names(ks) == [f"sha3_uniform_kernel<{L}>"], ks
        assert np.array_equal(got, got2)


@case
def cshake_chain_cut(ctx):
    """uniform ragged cSHAKE: device histogram (one bin: no scatter), then the cut; D224 (172-byte rate) is never cut"""
    n = chain_n(ctx)
    for d in (224, 256, 384, 512):
        L = KMAC_LANES[d]
        rnd = np.random.default_rng(d)
        data, off = ragged(rnd, np.full(n, 12 * KMAC_RATE[d] + 3))
        data_g = Guarded(ctx, len(data), 1, data, seed=d)
        off_t = dev_off(ctx, off)
        outs = []
        for env in (None, "1"):
            if env:
                ctx.mp.setenv("CAPY_NO_CHAIN_SPLIT", env)
            out_g = Guarded(ctx, n * 40, 1, seed=d + 1)
            ks = ctx.launched(lambda: cshake_dev(ctx, d, data_g, off_t, n, b"", b"Email Signature", 320, out_g))
            outs.append(out_g.get().reshape(n, 40))
            absent(ks, "len_scatter_kernel")
            if env or d == 224:
                assert names(ks)[-1] == f"sponge_kernel<{L}>", ks
                absent(ks, f"sponge_chain_kernel<{L}>")
            else:
                assert_chain(ks, L, n)
        ctx.mp.delenv("CAPY_NO_CHAIN_SPLIT")
        assert np.array_equal(outs[0], outs[1])
        idx = sample(n, d)
        want = ctx.orc.cshake_batch(*sub(data, off, idx), 320, b"", b"Email Signature", d, threads=0)
        assert np.array_equal(outs[0][idx], want), mismatch(outs[0][idx], want)


@case
def shake_plain_tiered_chain(ctx):
    """FIPS SHAKE128 (21 lanes) and SHAKE256 (17 lanes) through the plain, tiered and cut launches (hashlib reference)"""
    for bits, L in ((128, 21), (256, 17)):
        rate = 200 - bits // 4
        rnd = np.random.default_rng(bits)
        shapes = [("plain", rnd.integers(0, 500, size=300)), ("tiered", chain_bound(rnd, rate)),
                  ("chain", np.full(chain_n(ctx), 12 * rate + 1))]
        for mode, lens in shapes:
            data, off = ragged(rnd, lens)
            n = len(lens)
            out_bytes = 61
            data_g = Guarded(ctx, len(data), 1, data, seed=bits)
            off_t = dev_off(ctx, off)
            out_g = Guarded(ctx, n * out_bytes, 1, seed=bits + 1)
            ks = ctx.launched(lambda: ctx.call("capy_fips_shake_batch_dev", bits, data_g.ptr, off_t.data_ptr(), n,
                                               out_bytes, out_g.ptr))
            if mode == "tiered":
                only(ks, f"sponge_tiered_kernel<{L}>")
            elif mode == "chain":
                assert_chain(ks, L, n)
            else:
                assert names(ks)[-1] == f"sponge_kernel<{L}>", ks
            got = out_g.get().reshape(n, out_bytes)
            for i in sample(n, bits, k=200):
                m = data[int(off[i]):int(off[i + 1])].tobytes()
                h = hashlib.shake_128(m) if bits == 128 else hashlib.shake_256(m)
                assert got[i].tobytes() == h.digest(out_bytes), (mode, i)


# =========================================================================================================================
# KMACXOF
# =========================================================================================================================
@case
def kmac_tiered_all_d(ctx):
    """chain-bound KMACXOF (item D384 -> sponge_tiered_kernel<19>) at odd key, message and output addresses"""
    for d in (224, 256, 384, 512):
        rnd = np.random.default_rng(42 + d)
        lens = np.concatenate([[150_000, 99_999, 64_007, 168 * 500, 136 * 700 - 3, 172 * 400, 152 * 300 + 1],
                               rnd.integers(0, 300, size=2000)]).astype(np.int64)
        rnd.shuffle(lens)
        data, off = ragged(rnd, lens)
        n = len(lens)
        keys, koff = ragged(rnd, rnd.choice([0, 1, 32, 56, 200], size=n))
        data_g = Guarded(ctx, len(data), 1, data, seed=d)
        keys_g = Guarded(ctx, len(keys), 3, keys, seed=d + 1)
        off_t, koff_t = dev_off(ctx, off), dev_off(ctx, koff)
        out_g = Guarded(ctx, n * 61, 1, seed=d + 2)
        ks = ctx.launched(lambda: kmac_dev(ctx, d, keys_g, koff_t, data_g, off_t, n, b"My Tagged Application", 488, out_g))
        assert only(ks, f"sponge_tiered_kernel<{KMAC_LANES[d]}>")[0].block == (384, 1, 1), ks
        got = out_g.get().reshape(n, 61)
        want = ctx.orc.kmac_xof_batch(keys, koff, data, off, 488, b"My Tagged Application", d, threads=0)
        assert np.array_equal(got, want), (d, mismatch(got, want))


@case
def kmac_out_off_squeeze(ctx):
    """variable-length squeeze (out_off): a 1-byte and an empty output, the last item's bytes end at the guard"""
    for d in (224, 512):
        rnd = np.random.default_rng(d)
        n = 257
        data, off = ragged(rnd, rnd.integers(0, 400, size=n))
        keys, koff = ragged(rnd, np.full(n, 32))
        olens = rnd.integers(0, 700, size=n)
        olens[0], olens[1], olens[-1] = 1, 0, 1
        out_off = np.zeros(n + 1, np.uint64)
        out_off[1:] = np.cumsum(olens)
        data_g, keys_g = Guarded(ctx, len(data), 1, data), Guarded(ctx, len(keys), 1, keys)
        out_g = Guarded(ctx, int(out_off[-1]), 1)
        off_t, koff_t, oo_t = dev_off(ctx, off), dev_off(ctx, koff), dev_off(ctx, out_off)
        ks = ctx.launched(lambda: kmac_dev(ctx, d, keys_g, koff_t, data_g, off_t, n, b"", 0, out_g, oo_t))
        only(ks, f"sponge_kernel<{KMAC_LANES[d]}>")
        got = out_g.get()
        full = ctx.orc.kmac_xof_batch(keys, koff, data, off, 8 * int(olens.max()), b"", d, threads=0)
        for i in range(n):
            assert got[int(out_off[i]):int(out_off[i + 1])].tobytes() == full[i, :olens[i]].tobytes(), (d, i)


def kmac_fixed_case(ctx, d, n, key_len, key_stride, msg_len, msg_stride, out_bytes, offs=(1, 1, 1), seed=0):
    rnd = np.random.default_rng(seed)
    keys = rnd.integers(0, 256, size=max((n - 1) * key_stride + key_len, 1), dtype=np.uint8)
    keys_g = Guarded(ctx, len(keys), offs[0], keys, seed=seed)
    data = rnd.integers(0, 256, size=(n - 1) * msg_stride + msg_len, dtype=np.uint8) if msg_len else None
    data_g = Guarded(ctx, len(data), offs[1], data, seed=seed + 1) if msg_len else None
    out_g = Guarded(ctx, n * out_bytes, offs[2], seed=seed + 2)
    cs = b"KMAC fixed"
    s = np.frombuffer(cs, np.uint8)
    ks = ctx.launched(lambda: ctx.call("capy_kmac_xof_batch_fixed_dev", d, keys_g.ptr, key_len, key_stride,
                                       data_g.ptr if data_g else None, msg_len, msg_stride, n, s.ctypes.data, len(cs),
                                       8 * out_bytes, out_g.ptr))
    got = out_g.get().reshape(n, out_bytes)
    idx = sample(n, seed)
    kd, ko = rows(keys, key_len, key_stride, idx)
    md, mo = rows(data, msg_len, msg_stride, idx) if msg_len else (np.zeros(1, np.uint8), np.zeros(len(idx) + 1, np.uint64))
    want = ctx.orc.kmac_xof_batch(kd, ko, md, mo, 8 * out_bytes, cs, d, threads=0)
    assert np.array_equal(got[idx], want), (d, mismatch(got[idx], want))
    return ks, got


@case
def kmac_fixed_shapes(ctx):
    """two key blocks, strides beyond the lengths, msg_len = 0 with no data pointer, odd output length on a cut batch"""
    for d in (224, 256, 384, 512):
        L = KMAC_LANES[d]
        ks, _ = kmac_fixed_case(ctx, d, 513, 200, 203, 77, 85, 61, seed=d)  # key >= w: two key blocks
        assert names(ks)[-1] == f"sponge_kernel<{L}>", ks
        ks, _ = kmac_fixed_case(ctx, d, 300, 32, 40, 0, 0, 56, offs=(1, 0, 1), seed=d + 1)  # keygen shape
        assert names(ks)[-1] == f"sponge_kernel<{L}>", ks
    n = chain_n(ctx)
    for d in (256, 384, 512):
        L = KMAC_LANES[d]
        ks, got = kmac_fixed_case(ctx, d, n, 200, 203, 12 * KMAC_RATE[d] + 1, 12 * KMAC_RATE[d] + 9, 61, seed=d + 2)
        assert names(ks) == [f"sponge_chain_kernel<{L}>"], ks
        assert_chain(ks, L, n)
        ctx.mp.setenv("CAPY_NO_CHAIN_SPLIT", "1")
        ks, got2 = kmac_fixed_case(ctx, d, n, 200, 203, 12 * KMAC_RATE[d] + 1, 12 * KMAC_RATE[d] + 9, 61, seed=d + 2)
        ctx.mp.delenv("CAPY_NO_CHAIN_SPLIT")
        assert names(ks) == [f"sponge_kernel<{L}>"], ks
        assert np.array_equal(got, got2)


@case
def cshake_prefix_state(ctx):
    """a customisation string new to the ctx builds its prefix state once (prefix_state_kernel); D224's 172-byte
    bytepad width is not lane-aligned and has no cached state"""
    from capycrypt_b200 import Engine

    eng = Engine()
    try:
        rnd = np.random.default_rng(5)
        data, off = ragged(rnd, rnd.integers(0, 300, size=100))
        data_g, off_t = Guarded(ctx, len(data), 1, data), dev_off(ctx, off)
        for d, want_k in ((512, "prefix_state_kernel<17>"), (384, "prefix_state_kernel<19>"),
                          (256, "prefix_state_kernel<21>"), (224, None)):
            outs = []
            for rep in range(2):
                out_g = Guarded(ctx, 100 * 32, 1, seed=rep)
                ks = ctx.launched(lambda: cshake_dev(ctx, d, data_g, off_t, 100, b"fn", b"matrix prefix", 256, out_g,
                                                     eng=eng))
                if want_k and rep == 0:
                    assert names(ks)[0] == want_k, ks
                else:
                    assert not [k for k in names(ks) if k.startswith("prefix_state_kernel")], ks
                outs.append(out_g.get().reshape(100, 32))
            want = ctx.orc.cshake_batch(data, off, 256, b"fn", b"matrix prefix", d, threads=0)
            assert np.array_equal(outs[0], want) and np.array_equal(outs[1], want), d
    finally:
        eng.close()


# =========================================================================================================================
# authenticated encryption: the seal as one launch of two jobs, the open as dependent jobs
# =========================================================================================================================
class AeBatch:
    def __init__(self, ctx, d, n, max_len, seed, nonce_len=16):
        rnd = np.random.default_rng(seed)
        self.d, self.n, self.nonce_len = d, n, nonce_len
        self.msgs, self.off = ragged(rnd, rnd.integers(0, max_len, size=n))
        self.pws, self.poff = ragged(rnd, rnd.integers(0, 40, size=n))
        self.nonces = rnd.integers(0, 256, size=n * nonce_len, dtype=np.uint8)
        self.msgs_g = Guarded(ctx, len(self.msgs), 1, self.msgs, seed=seed)
        self.pws_g = Guarded(ctx, len(self.pws), 3, self.pws, seed=seed + 1)
        self.nonces_g = Guarded(ctx, len(self.nonces), 5, self.nonces, seed=seed + 2)
        self.off_t, self.poff_t = dev_off(ctx, self.off), dev_off(ctx, self.poff)

    def item(self, i):
        m = self.msgs[int(self.off[i]):int(self.off[i + 1])].tobytes()
        pw = self.pws[int(self.poff[i]):int(self.poff[i + 1])].tobytes()
        z = self.nonces[i * self.nonce_len:(i + 1) * self.nonce_len].tobytes()
        return m, pw, z

    def encrypt(self, ctx):
        ct_g = Guarded(ctx, len(self.msgs), 7, seed=1)
        tag_g = Guarded(ctx, self.n * 64, 1, seed=2)
        ks = ctx.launched(lambda: ctx.call("capy_sponge_encrypt_batch_dev", self.d, 0, self.pws_g.ptr, self.poff_t.data_ptr(),
                                           len(self.pws), self.nonces_g.ptr, self.nonce_len, self.msgs_g.ptr,
                                           self.off_t.data_ptr(), self.n, ct_g.ptr, tag_g.ptr))
        ct, tag = ct_g.get(), tag_g.get().reshape(self.n, 64)
        for i in sample(self.n, self.d, k=120):
            m, pw, z = self.item(i)
            c_ref, t_ref = R.sha3_encrypt(m, pw, self.d, z)
            assert ct[int(self.off[i]):int(self.off[i + 1])].tobytes() == c_ref and tag[i].tobytes() == t_ref, (self.d, i)
        return ks, ct, tag

    def decrypt(self, ctx, ct, tag, tamper):
        tag = tag.copy()
        tag[tamper, 0] ^= 1
        ct_g = Guarded(ctx, len(ct), 1, ct, seed=3)
        tag_g = Guarded(ctx, tag.size, 3, tag, seed=4)
        out_g = Guarded(ctx, len(ct), 5, seed=5)
        ok_g = Guarded(ctx, self.n, 1, seed=6)
        ks = ctx.launched(lambda: ctx.call("capy_sponge_decrypt_batch_dev", self.d, 0, self.pws_g.ptr, self.poff_t.data_ptr(),
                                           len(self.pws), self.nonces_g.ptr, self.nonce_len, ct_g.ptr, self.off_t.data_ptr(),
                                           tag_g.ptr, self.n, out_g.ptr, ok_g.ptr))
        out, ok = out_g.get(), ok_g.get()
        want_ok = np.ones(self.n, np.uint8)
        want_ok[tamper] = 0
        assert np.array_equal(ok, want_ok), np.nonzero(ok != want_ok)[0][:10]
        want = self.msgs.copy()
        for i in tamper:  # a failed item gets its ciphertext back
            want[int(self.off[i]):int(self.off[i + 1])] = ct[int(self.off[i]):int(self.off[i + 1])]
        assert np.array_equal(out, want)
        return ks


@case
def ae_seal_pair_launch(ctx):
    """sponge_kernel2: tag and keystream passes of the seal as one launch, ciphertext and tags at odd addresses"""
    for d in (224, 256, 384, 512):
        ae = AeBatch(ctx, d, 300, 600, seed=d)
        ks, ct, tag = ae.encrypt(ctx)
        only(ks, "ae_concat_kernel")
        only(ks, f"sponge_kernel2<{KMAC_LANES[d]}>")
        # a small open runs the two passes one after the other
        ks = ae.decrypt(ctx, ct, tag, tamper=[0, 17, 299])
        assert names(ks)[-3:] == [f"sponge_kernel<{KMAC_LANES[d]}>"] * 2 + ["ae_finish_kernel"], ks


def dep_threshold(sm):
    """smallest batch whose open runs as dependent jobs: ceil(n / 128) >= 3 x SMs"""
    return 128 * (3 * sm - 1) + 1


@case
def ae_open_dependent_jobs(ctx):
    """the open of a large batch is one sponge_chain_kernel launch whose second job reads what the first wrote (a
    partial last block); D224 (172-byte rate) runs two launches"""
    n = dep_threshold(ctx.sm) + 1
    for d in (224, 256, 384, 512):
        L = KMAC_LANES[d]
        ae = AeBatch(ctx, d, n, 48, seed=d)
        _, ct, tag = ae.encrypt(ctx)
        ks = ae.decrypt(ctx, ct, tag, tamper=[0, 5, n - 2, n - 1])
        if d == 224:
            absent(ks, "sponge_chain_kernel<21>")
            assert names(ks)[-3:] == ["sponge_kernel<21>"] * 2 + ["ae_finish_kernel"], ks
        else:
            assert_chain(ks, L, n)


@case
def ae_open_at_the_threshold(ctx):
    t = dep_threshold(ctx.sm)
    for n, cut in ((t, True), (t + 1, True), (t - 128, False)):
        ae = AeBatch(ctx, 512, n, 24, seed=n)
        _, ct, tag = ae.encrypt(ctx)
        ks = ae.decrypt(ctx, ct, tag, tamper=[1, n - 1])
        if cut:
            assert_chain(ks, 17, n)
        else:
            absent(ks, "sponge_chain_kernel<17>")
            assert names(ks)[-3:] == ["sponge_kernel<17>"] * 2 + ["ae_finish_kernel"], ks


# =========================================================================================================================
# Ed448
# =========================================================================================================================
R_ORDER = 2**446 - 13818066809895115352007386748515426880336692474882178609894547503885


def off_curve(pub112: bytes) -> bytes:
    b = bytearray(pub112)
    b[60] ^= 0x10
    assert not E.on_curve(E.point_from_bytes(bytes(b)))
    return bytes(b)


@case
def ed448_fixed_base_fresh_ctx(ctx):
    """the first fixed-base call of a ctx builds the comb table (fb_table_kernel); later calls reuse it"""
    from capycrypt_b200 import Engine

    eng = Engine()
    try:
        rnd = np.random.default_rng(1)
        n = 300
        sc = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
        want = ctx.orc.fixed_base_batch(sc, threads=0)
        sc_g = Guarded(ctx, len(sc), 1, sc)
        for rep in range(2):
            out_g = Guarded(ctx, n * 112, 1 + 2 * rep, seed=rep)
            ks = ctx.launched(lambda: eng._check(eng.lib.capy_ed448_fixed_base_batch_dev(eng._ctx, 0, ctx.stream, sc_g.ptr,
                                                                                          n, out_g.ptr)))
            want_k = ["scalar_prep_kernel", "fixed_base_kernel", "to_affine_kernel<16>"]
            assert names(ks) == (["scalar_prep_kernel", "fb_table_kernel"] + want_k[1:] if rep == 0 else want_k), ks
            got = out_g.get().reshape(n, 112)
            assert np.array_equal(got, want), mismatch(got, want)
    finally:
        eng.close()


@case
def ed448_var_base_off_curve_in_shared_inversion(ctx):
    """an off-curve point in a batch where to_affine inverts 16 items per thread: its row is zero, the flag is set, and
    the 15 items that share its inversion are exact"""
    n = 16 * 128 * 2  # 256 threads of 16 items, item i in thread i % 256
    rnd = np.random.default_rng(2)
    sc = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
    base = ctx.orc.fixed_base_batch(rnd.integers(0, 256, size=n * 56, dtype=np.uint8), threads=0)
    pts = base.copy()
    bad = 5 + 256 * 7
    pts[bad] = np.frombuffer(off_curve(pts[bad].tobytes()), np.uint8)
    rc, want = ctx.orc.var_base_batch(sc, pts, threads=0)
    want[bad] = 0
    sc_g, pts_g = Guarded(ctx, len(sc), 1, sc), Guarded(ctx, pts.size, 3, pts)
    out_g = Guarded(ctx, n * 112, 1)
    flag = ctx.torch.zeros(1, dtype=ctx.torch.int32, device="cuda")
    ks = ctx.launched(lambda: ctx.call("capy_ed448_var_base_batch_dev", sc_g.ptr, pts_g.ptr, n, out_g.ptr, flag.data_ptr()))
    assert names(ks) == ["var_base_kernel", "to_affine_kernel<16>", "any_bad_kernel"], ks
    assert ks[1].grid == (2, 1, 1), ks  # 256 threads of 16 items: rows bad % 256 + 256 k share one inversion
    got = out_g.get().reshape(n, 112)
    assert int(flag.item()) != 0
    assert not got[bad].any()
    assert np.array_equal(got, want), mismatch(got, want)


@case
def ed448_keygen_sign_verify_odd(ctx):
    """keygen, sign and verify with every byte buffer at an odd address; one off-curve key in a verify batch"""
    d = 256
    n = 16 * 128 * 2
    rnd = np.random.default_rng(3)
    pws, poff = ragged(rnd, rnd.integers(0, 40, size=n))
    msgs, moff = ragged(rnd, rnd.integers(0, 300, size=n))
    pws_g, msgs_g = Guarded(ctx, len(pws), 1, pws), Guarded(ctx, len(msgs), 3, msgs)
    poff_t, moff_t = dev_off(ctx, poff), dev_off(ctx, moff)
    pub_g = Guarded(ctx, n * 112, 1)
    ks = ctx.launched(lambda: ctx.call("capy_ed448_keygen_batch_dev", d, pws_g.ptr, poff_t.data_ptr(), n, pub_g.ptr))
    # (fb_table_kernel too when this is the engine's first fixed-base call)
    assert [k for k in names(ks) if k != "fb_table_kernel"][-3:] == ["scalar_prep_kernel", "fixed_base_kernel",
                                                                      "to_affine_kernel<16>"], ks
    pub = pub_g.get().reshape(n, 112)
    want = ctx.orc.keygen_batch(pws, poff, d, threads=0)
    assert np.array_equal(pub, want), mismatch(pub, want)
    h_g, z_g = Guarded(ctx, n * 56, 5), Guarded(ctx, n * 56, 7)
    ks = ctx.launched(lambda: ctx.call("capy_ed448_sign_batch_dev", d, pws_g.ptr, poff_t.data_ptr(), msgs_g.ptr,
                                       moff_t.data_ptr(), n, h_g.ptr, z_g.ptr))
    assert names(ks)[-1] == "sign_finish_kernel", ks
    h, z = h_g.get().reshape(n, 56), z_g.get().reshape(n, 56)
    ho, zo = ctx.orc.sign_batch(pws, poff, msgs, moff, d, threads=0)
    assert np.array_equal(h, ho) and np.array_equal(z, zo)
    bad = 9 + 256 * 3
    pub_bad = pub.copy()
    pub_bad[bad] = np.frombuffer(off_curve(pub[bad].tobytes()), np.uint8)
    h_bad = h.copy()
    h_bad[11, 0] ^= 1  # and one plain forgery
    for p, hh, flag_want in ((pub, h, 0), (pub_bad, h_bad, 1)):
        pg, hg, zg = Guarded(ctx, p.size, 1, p), Guarded(ctx, hh.size, 3, hh), Guarded(ctx, z.size, 5, z)
        ok_g = Guarded(ctx, n, 1)
        flag = ctx.torch.zeros(1, dtype=ctx.torch.int32, device="cuda")
        ks = ctx.launched(lambda: ctx.call("capy_ed448_verify_batch_dev", d, pg.ptr, msgs_g.ptr, moff_t.data_ptr(), hg.ptr,
                                           zg.ptr, n, ok_g.ptr, flag.data_ptr()))
        assert names(ks)[-1] == "verify_compare_kernel", ks
        ok = ok_g.get()
        want_ok = ctx.orc.verify_batch(p, msgs, moff, hh, z, d, threads=0)
        if flag_want:
            assert want_ok[bad] == 0 and want_ok[11] == 0
        assert np.array_equal(ok, want_ok), np.nonzero(ok != want_ok)[0][:10]
        assert int(flag.item() != 0) == flag_want


@case
def ed448_key_encrypt_decrypt_odd(ctx):
    """ECDHIES at odd addresses (one off-curve key: W.x = 0, flag set); decrypt with one wrong password"""
    d = 512
    rnd = np.random.default_rng(4)
    n = 5
    pws, poff = ragged(rnd, np.full(n, 16))
    pub = ctx.orc.keygen_batch(pws, poff, d)
    msgs, moff = ragged(rnd, [0, 17, 136, 700, 333])
    k = rnd.integers(0, 256, size=n * 56, dtype=np.uint8)
    bad = 3
    pub[bad] = np.frombuffer(off_curve(pub[bad].tobytes()), np.uint8)
    pub_g, k_g, msgs_g = Guarded(ctx, pub.size, 1, pub), Guarded(ctx, k.size, 3, k), Guarded(ctx, len(msgs), 5, msgs)
    moff_t = dev_off(ctx, moff)
    ct_g, tag_g, z_g = Guarded(ctx, len(msgs), 1), Guarded(ctx, n * 56, 3), Guarded(ctx, n * 112, 5)
    flag = ctx.torch.zeros(1, dtype=ctx.torch.int32, device="cuda")
    ks = ctx.launched(lambda: ctx.call("capy_ed448_key_encrypt_batch_dev", d, pub_g.ptr, k_g.ptr, msgs_g.ptr, moff_t.data_ptr(),
                                       n, ct_g.ptr, tag_g.ptr, z_g.ptr, flag.data_ptr()))
    only(ks, "sponge_kernel2<17>")
    assert names(ks)[-1] == "any_bad_kernel", ks
    ct, tag, zp = ct_g.get(), tag_g.get().reshape(n, 56), z_g.get().reshape(n, 112)
    assert int(flag.item()) != 0
    for i in range(n):
        if i == bad:
            continue
        m = msgs[int(moff[i]):int(moff[i + 1])].tobytes()
        c_ref, t_ref, z_ref = E.key_encrypt(E.point_from_bytes(pub[i].tobytes()), m, d, k[56 * i:56 * i + 56].tobytes())
        assert ct[int(moff[i]):int(moff[i + 1])].tobytes() == c_ref and tag[i].tobytes() == t_ref, i
        assert zp[i].tobytes() == E.point_to_bytes(z_ref), i
    pws2 = pws.copy()
    pws2[int(poff[1])] ^= 1
    good = [i for i in range(n) if i != bad]
    sel = np.array(good)
    pw_s, po_s = sub(pws2, poff, sel)
    m_s, mo_s = sub(msgs, moff, sel)
    c_s, _ = sub(ct, moff, sel)
    pw_g, z2_g, c_g, t_g = (Guarded(ctx, len(pw_s), 1, pw_s), Guarded(ctx, len(sel) * 112, 3, zp[sel]),
                            Guarded(ctx, len(c_s), 5, c_s), Guarded(ctx, len(sel) * 56, 7, tag[sel]))
    po_t, mo_t = dev_off(ctx, po_s), dev_off(ctx, mo_s)
    out_g, ok_g = Guarded(ctx, len(c_s), 1), Guarded(ctx, len(sel), 3)
    flag.zero_()
    ks = ctx.launched(lambda: ctx.call("capy_ed448_key_decrypt_batch_dev", d, pw_g.ptr, po_t.data_ptr(), z2_g.ptr, c_g.ptr,
                                       mo_t.data_ptr(), t_g.ptr, len(sel), out_g.ptr, ok_g.ptr, flag.data_ptr()))
    assert names(ks)[-2:] == ["ae_finish_kernel", "any_bad_kernel"], ks
    out, ok = out_g.get(), ok_g.get()
    assert ok.tolist() == [0 if i == 1 else 1 for i in good] and int(flag.item()) == 0
    want = m_s.copy()
    want[int(mo_s[1]):int(mo_s[2])] = c_s[int(mo_s[1]):int(mo_s[2])]
    assert np.array_equal(out, want)


# =========================================================================================================================
@pytest.fixture
def ctx(engine, oracle, tmp_path, monkeypatch):
    monkeypatch.delenv("CAPY_NO_CHAIN_SPLIT", raising=False)
    engine.set_plan_cache(False)  # every ragged call plans its own launch (the launches are what the cases check)
    return Ctx(engine, oracle, tmp_path, monkeypatch)


@pytest.mark.parametrize("name", list(CASES))
def test_launch_path(ctx, name):
    CASES[name](ctx)
    PASSED.add(name)


def test_every_kernel_ran_under_a_check():
    """the cases above, all run and passed in this session, launched every kernel of the library"""
    not_run = sorted(set(CASES) - PASSED)
    assert not not_run, f"coverage needs every case of this file to pass in the same session; missing: {not_run}"
    missing = sorted(KERNELS - SEEN)
    extra = sorted(SEEN - KERNELS)
    print(f"kernel coverage: {len(KERNELS & SEEN)}/{len(KERNELS)}")
    assert not missing, f"kernels no case launched: {missing}"
    assert not extra, f"kernels missing from KERNELS: {extra}"
