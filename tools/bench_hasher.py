"""Resumable streams against one-shot batches on one GPU, and host-fed updates against the link ceiling.

    python tools/bench_hasher.py [--out profiles/r03_hasher.json] [--reps 5]

device-resident, CUDA events, one warm-up pass of every shape:
  SHA3-256 and KMACXOF256 (D512, 32-byte keys, S = "My Tagged Application", 512-bit output) over 2^16 streams fed
  16 updates of 4 KiB each, then final  vs  the same data as 2^16 one-shot 64 KiB messages (capy_*_batch_dev)
host-fed: 2^12 SHA3-256 streams, one update of 1 MiB pieces from pinned memory through capy_hasher_update (host clock
around the blocking call) against capy_copy_probe's ceiling for the same bytes.
The hasher outputs are compared with the one-shot outputs (all items) outside the timed regions.  The card's name and
power limit are read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_hasher.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from capycrypt_b200.engine import Engine

    assert torch.cuda.is_available(), "needs a CUDA device"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    eng = Engine()
    n, updates, piece = 1 << 16, 16, 4096
    tag = b"My Tagged Application"
    g = torch.Generator(device="cuda")
    g.manual_seed(5)
    data = torch.randint(0, 256, (n, updates * piece), dtype=torch.uint8, device="cuda", generator=g)
    pieces = [data[:, k * piece:(k + 1) * piece].contiguous() for k in range(updates)]
    p_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * piece
    w_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * (updates * piece)
    keys = torch.randint(0, 256, (n * 32,), dtype=torch.uint8, device="cuda", generator=g)
    k_off = np.arange(n + 1, dtype=np.uint64) * 32
    t_koff = torch.from_numpy(k_off.astype(np.int64)).cuda()
    h_keys = keys.cpu().numpy()

    def events(fn, reps):
        fn()  # warm-up
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts)), ts

    res = {"gpu": gpu, "streams": n, "updates": updates, "piece_bytes": piece}
    for op, d, ob in (("sha3_256", 256, 32), ("kmacxof256_d512", 512, 64)):
        one = torch.zeros(n, ob, dtype=torch.uint8, device="cuda")
        if op == "sha3_256":
            oneshot = lambda: eng.sha3_dev(data, w_off, 256, one)
            make = lambda: eng.sha3_hasher(n, 256)
        else:
            oneshot = lambda: eng.kmac_xof_dev(keys, t_koff, data, w_off, 512, tag, 512, one)
            make = lambda: eng.kmac_xof_hasher(h_keys, k_off, tag, 512)
        ms_one, ts_one = events(oneshot, args.reps)
        streamed = torch.zeros(n, ob, dtype=torch.uint8, device="cuda")
        hs = []

        def run():
            h = hs[-1]
            for t in pieces:
                h.update_dev(t, p_off)
            h.final_dev(streamed, ob * 8)

        ts_h = []
        for rep in range(args.reps + 1):  # the first pass warms up; hashers are made outside the timed region
            hs.append(make())
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            torch.cuda.synchronize()
            if rep:
                ts_h.append(a.elapsed_time(b))
            hs.pop().close()
        assert torch.equal(streamed, one), f"{op}: streamed != one-shot"
        ms_h = float(np.median(ts_h))
        res[op] = {"oneshot_ms": ms_one, "oneshot_runs_ms": ts_one, "hasher_ms": ms_h, "hasher_runs_ms": ts_h,
                   "ratio_oneshot_over_hasher": ms_one / ms_h,
                   "hasher_GBps": n * updates * piece / (ms_h * 1e-3) / 1e9}

    # host-fed updates from pinned memory
    n2, mib = 1 << 12, 1 << 20
    h_data = eng.pinned(n2 * mib)
    h_data[:] = np.random.default_rng(1).integers(0, 256, size=n2 * mib, dtype=np.uint8)
    h_off = np.arange(n2 + 1, dtype=np.uint64) * mib
    h_out = eng.pinned(64)
    ceiling_ms = eng.copy_probe(h_data, h_out[:0], reps=3)
    ts = []
    for rep in range(args.reps + 1):
        h = eng.sha3_hasher(n2, 256)
        t0 = time.perf_counter()
        h.update(h_data, h_off)
        ts.append((time.perf_counter() - t0) * 1e3)
        got = h.final()
        h.close()
    ts = ts[1:]
    want = eng.sha3(h_data, h_off, 256)
    assert np.array_equal(got, want), "host-fed hasher != one-shot"
    ms = float(np.median(ts))
    res["host_update_2^12x1MiB_pinned"] = {"update_ms": ms, "runs_ms": ts, "GBps": n2 * mib / (ms * 1e-3) / 1e9,
                                           "link_ceiling_ms": ceiling_ms,
                                           "link_ceiling_GBps": n2 * mib / (ceiling_ms * 1e-3) / 1e9,
                                           "fraction_of_link": ceiling_ms / ms}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    eng.close()


if __name__ == "__main__":
    main()
