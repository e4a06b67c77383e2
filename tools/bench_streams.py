"""Encryption and verification streams against the one-shot calls on one GPU.

    python tools/bench_streams.py [--out profiles/r03_streams.json] [--reps 5]

2^16 items x 16 updates of 4 KiB (_dev calls, device-resident), then final, against the one-shot _dev call on the same
64 KiB messages, CUDA events around each, one warm-up pass of every shape:
  sha3_encrypt at D512 (capy_sponge_encrypt_batch_dev), key_encrypt with a prepared key at D512
  (capy_ed448_key_encrypt_prepared_batch_dev) and verify with a prepared key at D512 (capy_ed448_verify_prepared_batch_dev).
The one-shot times include their key derivation and curve work; the stream times do not: stream creation (a blocking
host call, host clock) is reported on its own.  Stream outputs are compared with the one-shot outputs (all items)
outside the timed regions.  The card's name and power limit are read in the same run and written beside the numbers.
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_streams.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from capycrypt_b200.engine import Engine, pack

    assert torch.cuda.is_available(), "needs a CUDA device"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    eng = Engine()
    n, updates, piece, d = 1 << 16, 16, 4096, 512
    g = torch.Generator(device="cuda")
    g.manual_seed(6)
    data = torch.randint(0, 256, (n, updates * piece), dtype=torch.uint8, device="cuda", generator=g)
    pieces = [data[:, k * piece:(k + 1) * piece].contiguous() for k in range(updates)]
    flat = data.reshape(-1)
    p_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * piece
    w_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * (updates * piece)
    rnd = np.random.default_rng(6)
    pws, pw_off = pack([rnd.bytes(16) for _ in range(n)])
    nonces = rnd.bytes(512 * n)
    k_rand = rnd.bytes(56 * n)
    t_pws, t_pwo = torch.from_numpy(pws).cuda(), torch.from_numpy(pw_off.astype(np.int64)).cuda()
    t_nonce = torch.from_numpy(np.frombuffer(nonces, np.uint8).copy()).cuda()
    t_k = torch.from_numpy(np.frombuffer(k_rand, np.uint8).copy()).cuda()
    signer = b"bench signer"
    pub = eng.ed448_keygen(*pack([signer]), d)[0].tobytes()
    key = eng.ed448_pub_prepare(pub)
    assert key.uses_comb

    def timed(fn, reps):
        ts = []
        for rep in range(reps + 1):  # the first pass warms up
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            if rep:
                ts.append(a.elapsed_time(b))
        return float(np.median(ts)), ts

    def host_ms(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    res = {"gpu": gpu, "streams": n, "updates": updates, "piece_bytes": piece, "d": d}
    ct_one = torch.empty_like(flat)
    t_out = [torch.empty_like(p) for p in pieces]

    def stream_case(name, make, tag_bytes, oneshot, outputs):
        """tag_bytes = 0: a verification stream (final: n ok flags)"""
        ms_one, ts_one = timed(oneshot, args.reps)
        tag = torch.zeros(n, max(tag_bytes, 1), dtype=torch.uint8, device="cuda")
        create, ts = [], []
        for rep in range(args.reps + 1):  # streams are made outside the timed region
            ms_c, st = host_ms(make)
            create.append(ms_c)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for k, t in enumerate(pieces):
                if tag_bytes:
                    st.update_dev(t, p_off, t_out[k])
                else:
                    st.update_dev(t, p_off)
            st.final_dev(tag if tag_bytes else tag.reshape(-1))
            b.record()
            torch.cuda.synchronize()
            if rep:
                ts.append(a.elapsed_time(b))
            st.close()
        outputs(tag)
        ms = float(np.median(ts))
        res[name] = {"oneshot_ms": ms_one, "oneshot_runs_ms": ts_one, "stream_ms": ms, "stream_runs_ms": ts,
                     "ratio_oneshot_over_stream": ms_one / ms, "stream_GBps": n * updates * piece / (ms * 1e-3) / 1e9,
                     "create_ms_median": float(np.median(create[1:])), "create_runs_ms": create[1:]}

    def ct_of_stream():
        return torch.cat(t_out, dim=1).reshape(-1)

    # sha3_encrypt
    tag_one = torch.empty(n, 64, dtype=torch.uint8, device="cuda")

    def check_sponge(tag):
        assert torch.equal(ct_of_stream(), ct_one) and torch.equal(tag, tag_one), "sha3_encrypt: stream != one-shot"

    stream_case("sha3_encrypt_d512",
                lambda: eng.sponge_encrypt_stream(pws, pw_off, nonces, 512, d),
                64,
                lambda: eng.sponge_encrypt_dev(t_pws, t_pwo, len(pws), t_nonce, 512, flat, w_off, d, ct_one, tag_one),
                check_sponge)
    # key_encrypt, prepared key
    tag56 = torch.empty(n, 56, dtype=torch.uint8, device="cuda")
    z_one = torch.empty(n, 112, dtype=torch.uint8, device="cuda")

    def check_key(tag):
        assert torch.equal(ct_of_stream(), ct_one) and torch.equal(tag, tag56), "key_encrypt: stream != one-shot"

    stream_case("key_encrypt_prepared_d512",
                lambda: eng.ed448_key_encrypt_stream(key, k_rand, d)[0],
                56,
                lambda: eng.ed448_key_encrypt_prepared_dev(key, t_k, flat, w_off, d, ct_one, tag56, z_one),
                check_key)
    # verify, prepared key: signatures of the whole messages
    t_h = torch.empty(n, 56, dtype=torch.uint8, device="cuda")
    t_z = torch.empty(n, 56, dtype=torch.uint8, device="cuda")
    t_spw, t_spo = torch.from_numpy(np.frombuffer(signer * n, np.uint8).copy()).cuda(), \
        torch.arange(n + 1, dtype=torch.int64, device="cuda") * len(signer)
    eng.ed448_sign_dev(t_spw, t_spo, flat, w_off, d, t_h, t_z)
    torch.cuda.synchronize()
    h, z = t_h.cpu().numpy(), t_z.cpu().numpy()
    ok_one = torch.zeros(n, dtype=torch.uint8, device="cuda")

    def check_verify(ok):
        assert torch.equal(ok.reshape(-1), ok_one) and bool(ok_one.all()), "verify: stream != one-shot"

    stream_case("verify_prepared_d512",
                lambda: eng.ed448_verify_stream(key, h, z, d),
                0,
                lambda: eng.ed448_verify_prepared_dev(key, flat, w_off, t_h, t_z, d, ok_one),
                check_verify)
    key.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    eng.close()


if __name__ == "__main__":
    main()
