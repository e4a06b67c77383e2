"""Two-pass sign and decryption streams against the one-shot calls on one GPU.

    python tools/bench_two_pass_streams.py [--out profiles/r03_two_pass_streams.json] [--reps 5]

2^16 messages x 16 pieces of 4 KiB per pass at D512, against the one-shot call on the same 2^16 x 64 KiB messages:
sign (capy_ed448_sign_batch), sha3_decrypt (capy_sponge_decrypt_batch) and key_decrypt (capy_ed448_key_decrypt_batch).
  _dev path: device-resident pieces, CUDA events around pass 1, next_pass, pass 2 and the final; the one-shot _dev call
             likewise.  Stream creation (a blocking host call) is timed on its own, host clock.
  host path: the same bytes from pageable host memory through the host entry points, host clock, both passes and the
             final; the one-shot host call likewise.
The one-shot times include their key derivation and curve work; the stream times cover only what follows creation.
Keccak work per 136-byte block: a sign stream does 1 + 2 permutations, a decryption stream 2 + 2, the one-shot calls 2.
Outputs of every path are compared with the one-shot outputs outside the timed regions.  The card's name and power limit
are read in the same run.
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_two_pass_streams.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from capycrypt_b200.engine import Engine, pack

    assert torch.cuda.is_available(), "needs a CUDA device"
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    eng = Engine()
    n, ups, piece, d = 1 << 16, 16, 4096, 512
    g = torch.Generator(device="cuda")
    g.manual_seed(7)
    data = torch.randint(0, 256, (n, ups * piece), dtype=torch.uint8, device="cuda", generator=g)
    flat = data.reshape(-1)
    p_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * piece
    w_off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * (ups * piece)
    h_poff = p_off.cpu().numpy().astype(np.uint64)
    h_woff = w_off.cpu().numpy().astype(np.uint64)
    rnd = np.random.default_rng(7)
    pws, pw_off = pack([rnd.bytes(16) for _ in range(n)])
    nonces = rnd.bytes(512 * n)
    t_pws, t_pwo = torch.from_numpy(pws).cuda(), torch.from_numpy(pw_off.astype(np.int64)).cuda()
    t_nonce = torch.from_numpy(np.frombuffer(nonces, np.uint8).copy()).cuda()

    def events(fn):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b), r

    def host_ms(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3, r

    def runs(fn, clock):
        ts = [clock(fn)[0] for _ in range(args.reps + 1)][1:]  # the first run warms up
        return float(np.median(ts)), ts

    res = {"gpu": gpu, "messages": n, "pieces_per_pass": ups, "piece_bytes": piece, "d": d}

    def case(name, make, dev_passes, host_passes, oneshot_dev, oneshot_host, check):
        one_dev = runs(oneshot_dev, events)
        one_host = runs(oneshot_host, host_ms)
        create, dev_ts, host_ts = [], [], []
        for rep in range(args.reps + 1):
            ms_c, st = host_ms(make)
            ms_d, out_d = events(lambda: dev_passes(st))
            st.close()
            ms_c2, st = host_ms(make)
            ms_h, out_h = host_ms(lambda: host_passes(st))
            st.close()
            if rep == 0:
                check(out_d, out_h)
            else:
                create += [ms_c, ms_c2]
                dev_ts.append(ms_d)
                host_ts.append(ms_h)
        res[name] = {"oneshot_dev_ms": one_dev[0], "oneshot_dev_runs_ms": one_dev[1],
                     "stream_dev_ms": float(np.median(dev_ts)), "stream_dev_runs_ms": dev_ts,
                     "oneshot_host_ms": one_host[0], "oneshot_host_runs_ms": one_host[1],
                     "stream_host_ms": float(np.median(host_ts)), "stream_host_runs_ms": host_ts,
                     "ratio_dev_oneshot_over_stream": one_dev[0] / float(np.median(dev_ts)),
                     "create_ms_median": float(np.median(create)), "create_runs_ms": create}
        print(name, json.dumps(res[name]))

    pieces = [data[:, k * piece:(k + 1) * piece].contiguous() for k in range(ups)]
    h_pieces = [p.cpu().numpy().reshape(-1) for p in pieces]

    # ---- sign
    wh, wz = torch.empty(n, 56, dtype=torch.uint8, device="cuda"), torch.empty(n, 56, dtype=torch.uint8, device="cuda")
    h_msgs = flat.cpu().numpy()

    def sign_dev(st):
        for p in pieces:
            st.update_dev(p, p_off)
        st.next_pass_dev()
        for p in pieces:
            st.update_dev(p, p_off)
        h, z, ok = torch.empty_like(wh), torch.empty_like(wz), torch.empty(n, dtype=torch.uint8, device="cuda")
        st.final_dev(h, z, ok)
        return h, z, ok

    def sign_host(st):
        for p in h_pieces:
            st.update(p, h_poff)
        st.next_pass()
        for p in h_pieces:
            st.update(p, h_poff)
        return st.final()

    def sign_check(out_d, out_h):
        h, z, ok = out_d
        assert bool(ok.all()) and torch.equal(h, wh) and torch.equal(z, wz), "sign _dev stream != one-shot"
        hh, zz, okh = out_h
        assert okh.all() and np.array_equal(hh, wh.cpu().numpy()) and np.array_equal(zz, wz.cpu().numpy()), "sign host"

    case("sign_d512", lambda: eng.ed448_sign_stream(pws, pw_off, d), sign_dev, sign_host,
         lambda: eng.ed448_sign_dev(t_pws, t_pwo, flat, w_off, d, wh, wz),
         lambda: eng.ed448_sign(pws, pw_off, h_msgs, h_woff, d), sign_check)

    # ---- sha3_decrypt of the data encrypted once
    ct = torch.empty_like(flat)
    tag = torch.empty(n, 64, dtype=torch.uint8, device="cuda")
    eng.sponge_encrypt_dev(t_pws, t_pwo, len(pws), t_nonce, 512, flat, w_off, d, ct, tag)
    torch.cuda.synchronize()
    ct_pieces = [ct.reshape(n, -1)[:, k * piece:(k + 1) * piece].contiguous() for k in range(ups)]
    h_ct_pieces = [p.cpu().numpy().reshape(-1) for p in ct_pieces]
    h_ct, h_tag = ct.cpu().numpy(), tag.cpu().numpy()
    pt_one = torch.empty_like(flat)
    ok_one = torch.empty(n, dtype=torch.uint8, device="cuda")
    outs = [torch.empty_like(p) for p in ct_pieces]

    def dec_dev(st):
        for p in ct_pieces:
            st.update_dev(p, p_off)
        verdict = torch.empty(n, dtype=torch.uint8, device="cuda")
        st.next_pass_dev(verdict)
        for p, o in zip(ct_pieces, outs):
            st.decrypt_dev(p, p_off, o)
        ok = torch.empty(n, dtype=torch.uint8, device="cuda")
        st.final_dev(ok)
        return verdict, ok

    def dec_host(st):
        for p in h_ct_pieces:
            st.update(p, h_poff)
        _, verdict = st.next_pass()
        last = [st.decrypt(p, h_poff) for p in h_ct_pieces]
        _, ok = st.final()
        return verdict, ok, last

    def dec_check(out_d, out_h):
        v, ok = out_d
        assert bool(v.all()) and bool(ok.all()) and torch.equal(torch.cat(outs, 1).reshape(-1), flat), "decrypt _dev"
        vh, okh, last = out_h
        assert vh.all() and okh.all() and all(np.array_equal(a, b) for a, b in zip(last, h_pieces)), "decrypt host"

    case("sha3_decrypt_d512", lambda: eng.sponge_decrypt_stream(pws, pw_off, nonces, 512, h_tag, d), dec_dev, dec_host,
         lambda: eng.sponge_decrypt_dev(t_pws, t_pwo, len(pws), t_nonce, 512, ct, w_off, tag, d, pt_one, ok_one),
         lambda: eng.sponge_decrypt(pws, pw_off, nonces, 512, h_ct, h_woff, h_tag, d), dec_check)

    # ---- key_decrypt: one recipient password per message
    pubs = eng.ed448_keygen(pws, pw_off, d)
    k_rand = rnd.bytes(56 * n)
    t_pub = torch.from_numpy(pubs.reshape(-1).copy()).cuda()
    t_k = torch.from_numpy(np.frombuffer(k_rand, np.uint8).copy()).cuda()
    tag56 = torch.empty(n, 56, dtype=torch.uint8, device="cuda")
    z = torch.empty(n, 112, dtype=torch.uint8, device="cuda")
    eng.ed448_key_encrypt_dev(t_pub, t_k, flat, w_off, d, ct, tag56, z)
    torch.cuda.synchronize()
    ct_pieces[:] = [ct.reshape(n, -1)[:, k * piece:(k + 1) * piece].contiguous() for k in range(ups)]
    h_ct_pieces[:] = [p.cpu().numpy().reshape(-1) for p in ct_pieces]
    h_ct, h_tag56, h_z = ct.cpu().numpy(), tag56.cpu().numpy(), z.cpu().numpy()
    case("key_decrypt_d512", lambda: eng.ed448_key_decrypt_stream(pws, pw_off, h_z, h_tag56, d), dec_dev, dec_host,
         lambda: eng.ed448_key_decrypt_dev(t_pws, t_pwo, z, ct, w_off, tag56, d, pt_one, ok_one),
         lambda: eng.ed448_key_decrypt(pws, pw_off, h_z, h_ct, h_woff, h_tag56, d), dec_check)

    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    eng.close()


if __name__ == "__main__":
    main()
