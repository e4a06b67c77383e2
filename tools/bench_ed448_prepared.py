"""Prepared public keys against the per-item-key pipelines: verify against one signer and key_encrypt to one recipient.

    python tools/bench_ed448_prepared.py [--out profiles/r03_ed448_prepared.json] [--reps 5]

Workload: D512, 256-byte messages, one key from keygen.  For n = 2^18 and 2^20 it times, with CUDA events around the
device-resident `_dev` calls on torch's stream (after a warm-up call of each shape):
  verify       capy_ed448_verify_batch_dev with the key repeated n times   vs  capy_ed448_verify_prepared_batch_dev
  key_encrypt  capy_ed448_key_encrypt_batch_dev with the key repeated       vs  capy_ed448_key_encrypt_prepared_batch_dev
and the blocking capy_ed448_pub_prepare (median of several, host clock).  Outside the timed region the prepared outputs
are compared with the per-item-key outputs (all items) and with the oracle (a seeded sample with the first and the last
item).  The card's name and power limit are read in the same run and written beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info() -> dict:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in r.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ed448_prepared.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="18,20", help="log2 of the batch sizes")
    args = ap.parse_args()

    import torch

    from capycrypt_b200 import Engine
    from oracle import cpu
    from oracle import ref_ed448 as E

    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    eng, orc = Engine(), cpu.get()
    d, mlen = 512, 256
    pw = b"bench signer"
    pub = eng.ed448_keygen(np.frombuffer(pw, np.uint8), np.array([0, len(pw)], np.uint64), d)[0].tobytes()

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return statistics.median(ms), min(ms), max(ms)

    prep_ms = []
    for _ in range(7):
        t0 = time.perf_counter()
        k = eng.ed448_pub_prepare(pub)
        prep_ms.append((time.perf_counter() - t0) * 1e3)
        k.close()
    key = eng.ed448_pub_prepare(pub)
    assert key.uses_comb

    res = {"workload": f"D{d}, {mlen}-byte messages, one key from keygen", "gpu": gpu_info(),
           "prepare_ms": {"median": statistics.median(prep_ms), "min": min(prep_ms), "max": max(prep_ms),
                          "runs": len(prep_ms)},
           "timing": f"CUDA events around one _dev call, median of {args.reps} after one warm-up call", "sizes": {}}
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    rs = np.random.default_rng(3)
    for lg in (int(s) for s in args.sizes.split(",")):
        n = 1 << lg
        msg = torch.randint(0, 256, (n * mlen,), dtype=torch.uint8, device="cuda", generator=g)
        moff = torch.arange(n + 1, dtype=torch.int64, device="cuda") * mlen
        pws = torch.tensor(list(pw), dtype=torch.uint8, device="cuda").repeat(n)
        pw_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * len(pw)
        h = torch.zeros(n * 56, dtype=torch.uint8, device="cuda")
        z = torch.zeros(n * 56, dtype=torch.uint8, device="cuda")
        eng.ed448_sign_dev(pws, pw_off, msg, moff, d, h, z)
        h.view(n, 56)[1::2, 7] ^= 1  # every other signature is forged
        pubs = torch.tensor(list(pub), dtype=torch.uint8, device="cuda").repeat(n)
        ok0 = torch.zeros(n, dtype=torch.uint8, device="cuda")
        ok1 = torch.zeros(n, dtype=torch.uint8, device="cuda")
        v0 = timed(lambda: eng.ed448_verify_dev(pubs, msg, moff, h, z, d, ok0), args.reps)
        v1 = timed(lambda: eng.ed448_verify_prepared_dev(key, msg, moff, h, z, d, ok1), args.reps)

        kr = torch.randint(0, 256, (n * 56,), dtype=torch.uint8, device="cuda", generator=g)
        ct0, ct1 = (torch.zeros(n * mlen, dtype=torch.uint8, device="cuda") for _ in range(2))
        t0, t1 = (torch.zeros(n * 56, dtype=torch.uint8, device="cuda") for _ in range(2))
        z0, z1 = (torch.zeros(n * 112, dtype=torch.uint8, device="cuda") for _ in range(2))
        e0 = timed(lambda: eng.ed448_key_encrypt_dev(pubs, kr, msg, moff, d, ct0, t0, z0), args.reps)
        e1 = timed(lambda: eng.ed448_key_encrypt_prepared_dev(key, kr, msg, moff, d, ct1, t1, z1), args.reps)
        torch.cuda.synchronize()

        # outputs: prepared == per-item key (all items), and the oracle on a seeded sample with the first and last item
        assert torch.equal(ok0, ok1), "verify: prepared != per-item key"
        assert bool(ok1.view(-1)[0::2].all()) and not bool(ok1.view(-1)[1::2].any())
        assert torch.equal(ct0, ct1) and torch.equal(t0, t1) and torch.equal(z0, z1), "key_encrypt: prepared != per-item key"
        idx = np.array(sorted(set(rs.choice(n, size=200, replace=False).tolist()) | {0, n - 1}))
        m_np, h_np, z_np = msg.cpu().numpy().reshape(n, mlen), h.cpu().numpy().reshape(n, 56), z.cpu().numpy().reshape(n, 56)
        so = np.arange(len(idx) + 1, dtype=np.uint64) * mlen
        want = orc.verify_batch(np.frombuffer(pub * len(idx), np.uint8), m_np[idx].reshape(-1), so, h_np[idx].reshape(-1),
                                z_np[idx].reshape(-1), d, threads=0)
        assert np.array_equal(ok1.cpu().numpy()[idx], want), "verify: prepared != oracle"
        ct_np, t_np, zz_np, k_np = (ct1.cpu().numpy().reshape(n, -1), t1.cpu().numpy().reshape(n, 56),
                                    z1.cpu().numpy().reshape(n, 112), kr.cpu().numpy().reshape(n, 56))
        vp = E.point_from_bytes(pub)
        for i in idx[:8].tolist() + [n - 1]:
            c_ref, t_ref, z_ref = E.key_encrypt(vp, m_np[i].tobytes(), d, k_np[i].tobytes())
            assert ct_np[i].tobytes() == c_ref and t_np[i].tobytes() == t_ref and zz_np[i].tobytes() == E.point_to_bytes(z_ref)

        def row(t):
            return {"ms_median": t[0], "ms_min": t[1], "ms_max": t[2], "items_per_s": n / (t[0] * 1e-3)}

        res["sizes"][f"2^{lg}"] = {
            "verify_key_repeated": row(v0), "verify_prepared": row(v1), "verify_speedup": v0[0] / v1[0],
            "key_encrypt_key_repeated": row(e0), "key_encrypt_prepared": row(e1), "key_encrypt_speedup": e0[0] / e1[0],
            "oracle_sample": int(len(idx))}
        del msg, pws, h, z, pubs, ok0, ok1, kr, ct0, ct1, t0, t1, z0, z1
        torch.cuda.empty_cache()
    # break-even: the batch size from which preparing the key pays for itself within one call
    s18 = res["sizes"].get("2^18")
    if s18:
        for op in ("verify", "key_encrypt"):
            saved_ms_per_item = (s18[f"{op}_key_repeated"]["ms_median"] - s18[f"{op}_prepared"]["ms_median"]) / (1 << 18)
            res[f"{op}_break_even_items"] = res["prepare_ms"]["median"] / saved_ms_per_item if saved_ms_per_item > 0 else None
    key.close()
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
