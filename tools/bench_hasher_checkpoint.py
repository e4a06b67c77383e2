"""Export, import and fork of resumable streams on one GPU.

    python tools/bench_hasher_checkpoint.py [--out profiles/r03_hasher_checkpoint.json] [--reps 5]

Streams: 2^20 SHA3-256 and 2^16 KMACXOF256 (D256, 32-byte keys), each fed one 200-byte piece, so every stream is
mid-message (a carry of 64 or 32 bytes).
  export / import: the blob (64 + n (208 + rate) bytes) to and from pinned (capy_host_alloc) and pageable memory; host
    clock around the blocking call, median of --reps; GB/s of blob bytes against capy_copy_probe's ceiling for the same
    bytes in the same direction from the same kind of memory.  Import includes creating the hasher (cudaMalloc, memset).
  fork: identity and replicate-one (every item a copy of item 0) of the 2^20 SHA3-256 streams.  Whole call: CUDA events
    around the blocking call (it allocates and zeroes the new hasher and uploads the map).  Copy kernel: the
    sponge_chain_kernel time from torch.profiler in a separate pass.  GB/s of bytes read + written: per item the map
    entry (8 B) and the stream read and written (2 x (208 + rate) B), against the HBM3e data-sheet 7.7 TB/s.
Every exported blob is checked to import and export back to itself, and forks against their sources, outside the timed
regions.  The card's name and power limit are read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_GBS = 7700.0


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_hasher_checkpoint.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from capycrypt_b200 import _binding as B
    from capycrypt_b200.engine import Engine, pack

    assert torch.cuda.is_available(), "needs a CUDA device"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    eng = Engine()
    lib, ctx = eng.lib, eng._ctx
    rnd = np.random.default_rng(1)
    res = {"gpu": gpu, "export_import": [], "fork": []}

    def median_s(fn, reps):
        fn()  # warm-up
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts))

    def check(rc):
        if rc != B.OK:
            raise B.CapyError(rc, lib.capy_strerror(rc).decode())

    piece = 200
    for name, n, rate in (("SHA3-256", 1 << 20, 136), ("KMACXOF256", 1 << 16, 168)):
        if name == "SHA3-256":
            h = eng.sha3_hasher(n, 256)
        else:
            h = eng.kmac_xof_hasher(rnd.integers(0, 256, n * 32, dtype=np.uint8), np.arange(n + 1, dtype=np.uint64) * 32,
                                    b"", 256)
        h.update(rnd.integers(0, 256, n * piece, dtype=np.uint8), np.arange(n + 1, dtype=np.uint64) * piece)
        size = 64 + n * (208 + rate)
        ref = h.export()
        assert ref.size == size
        with eng.import_hasher(ref) as back:
            assert np.array_equal(back.export(), ref)
        for mem in ("pinned", "pageable"):
            blob = eng.pinned(size) if mem == "pinned" else np.empty(size, np.uint8)
            blob[:] = ref

            def export():
                check(lib.capy_hasher_export(ctx, h.handle, blob.ctypes.data, size))

            def imp():
                out = C.c_void_p()
                check(lib.capy_hasher_import(ctx, blob.ctypes.data, size, C.byref(out)))
                lib.capy_hasher_free(out)

            t_exp = median_s(export, args.reps)
            assert np.array_equal(blob, ref)
            t_imp = median_s(imp, args.reps)
            empty = np.zeros(0, np.uint8)
            d2h = eng.copy_probe(empty, blob, reps=args.reps) / 1e3
            h2d = eng.copy_probe(blob, empty, reps=args.reps) / 1e3
            for op, t, ceil in (("export", t_exp, d2h), ("import", t_imp, h2d)):
                res["export_import"].append({
                    "op": op, "streams": name, "n": n, "memory": mem, "blob_bytes": size, "ms": round(t * 1e3, 3),
                    "GBps": round(size / t / 1e9, 2), "link_ceiling_GBps": round(size / ceil / 1e9, 2),
                    "fraction_of_link": round(ceil / t, 3)})
                print(json.dumps(res["export_import"][-1]), flush=True)
        if name != "SHA3-256":
            h.close()
            continue
        # forks of the 2^20 SHA3-256 streams
        from torch.profiler import ProfilerActivity, profile

        for kind, src in (("identity", np.arange(n, dtype=np.uint64)), ("replicate one", np.zeros(n, np.uint64))):
            moved = n * (8 + 2 * (208 + rate))

            def fork():
                out = C.c_void_p()
                check(lib.capy_hasher_fork(ctx, h.handle, src.ctypes.data, n, C.byref(out)))
                lib.capy_hasher_free(out)

            fork()
            torch.cuda.synchronize()
            ts = []
            for _ in range(args.reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fork()
                b.record()
                b.synchronize()
                ts.append(a.elapsed_time(b) / 1e3)
            t_call = float(np.median(ts))
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                torch.zeros(1, device="cuda").add_(1)  # the profiler's first activity buffer
                torch.cuda.synchronize()
                fork()
                torch.cuda.synchronize()
            t_kern = sum(e.device_time_total for e in prof.key_averages() if "sponge_chain_kernel" in e.key) / 1e6
            with h.fork(src[:4]) as f:  # a fork of four: the same records as their sources
                rec = f.export()[64:].reshape(4, -1)
                srcs = ref[64:].reshape(n, -1)[src[:4].astype(np.int64)]
                assert np.array_equal(rec, srcs)
            res["fork"].append({
                "map": kind, "streams": "SHA3-256", "n": n, "bytes_read_written": moved, "call_ms": round(t_call * 1e3, 3),
                "call_GBps": round(moved / t_call / 1e9, 1), "kernel_ms": round(t_kern * 1e3, 4),
                "kernel_GBps": round(moved / t_kern / 1e9, 1) if t_kern else None,
                "kernel_fraction_of_hbm_datasheet": round(moved / t_kern / 1e9 / HBM_GBS, 3) if t_kern else None})
            print(json.dumps(res["fork"][-1]), flush=True)
        h.close()
    eng.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
