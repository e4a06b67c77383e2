#!/usr/bin/env python3
"""bench.py -- headline benchmark of the capyCRYPT B200 batch engine (contract: see the task brief).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): SHA3-256 GB/s (+ Ed448 scalar-mults/s in `extra`).  A step is one pass of the hot
path over one batch: SHA3-256 (SecParam::D256) over 2^20 random 64-byte messages per GPU
(BASELINE.json configs[0], the configuration the metric is quoted on).  Weak scaling: every rank hashes
its own 2^20-message batch, no collective on the data path; `value` = bytes hashed by all ranks / max
time over ranks.  Prints ONE JSON line on rank 0.

The oracle (oracle/) is touched only by the cpu_baseline leg and by --impl reference.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_MSGS = 1 << 20
MSG_LEN = 64
DIGEST = 32
N_ROT = 4  # rotating input/output buffers: 4 x (64 + 32) MiB = 384 MiB > 126 MB of L2
OPS_PER_PERM = 4320  # SURVEY.md 8d: 122 LOP3 + 58 SHF per round x 24
MAC_FIXED = 2.03e5  # canonical 32x32->64 MAC budgets per scalar multiplication (SURVEY.md 8d / App. D)
MAC_VAR = 7.12e5
# IMAD.WIDE instructions the kernels actually execute per scalar multiplication (SASS counts x trip counts, DESIGN.md 4):
# fixed base = 90 mixed additions x 7 M + dual isogeny + scalar glue on the isogenous curve; variable base =
# 448 x (4 S + 3 M) + 112 M + 113 x 9 M + table (1 dbl + 6 add), M = 193, S = 110
MAC_EXEC_FIXED = 1.23e5
MAC_EXEC_VAR = 6.86e5
WARP_TIER_US_PER_PERM = 2.04  # chain speed of the fastest tier (one warp per message), profiles/README.md
PEAK_FALLBACK = {"lop3": 18.52e12, "imad_wide": 8.67e12}  # profiles/r01_peaks_int_pipes.json
# --dump-outputs writes a fixed, seeded sample of the digests: all 2^20 x 32 bytes would be 128 MiB as float32
DUMP_ROWS = 1 << 18
DUMP_SEED = 0


def host_threads() -> int:
    """Host threads this process may use (the same call at every N: torchrun forces OMP_NUM_THREADS=1, which must
    not decide how many cores the CPU reference gets)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def workload_config() -> dict:
    """`config` of the JSON line -- the SAME dict in both arms (b200 and reference)."""
    return {"workload": "sha3_256_2^20x64B", "per_gpu_msgs": N_MSGS, "msg_bytes": MSG_LEN, "sec_param": "D256",
            "l2": f"inputs/outputs rotate over {N_ROT} buffer pairs (384 MiB per GPU > 126 MB L2)",
            "sharding": "one 2^20-message batch per rank, no collective"}


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------------------------------------------
# clocks: sample SM clock + throttle reasons DURING the timed region (NVML, same data as nvidia-smi)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int, period_s: float = 0.02):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)
        self.period = period_s

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        s = sorted(self.samples)
        return {
            "sm_mhz": s[len(s) // 2] if s else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples": len(s),
        }


# ------------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) -- the ONLY place bench.py touches oracle/
# ------------------------------------------------------------------------------------------------------
def _time_sha3(orc, n, threads, lean, budget_s, rate_hint=None):
    """GB/s of oracle.sha3_batch over n x 64 B messages, repeated for about budget_s."""
    import numpy as np

    rng = np.random.default_rng(1)
    buf = rng.integers(0, 256, size=n * MSG_LEN, dtype=np.uint8)
    off = np.arange(n + 1, dtype=np.uint64) * MSG_LEN
    orc.sha3_batch(buf, off, 256, threads=threads, lean=lean)  # warm
    t0 = time.perf_counter()
    orc.sha3_batch(buf, off, 256, threads=threads, lean=lean)
    rate = n / (time.perf_counter() - t0)
    reps = max(1, int(rate * budget_s / n))
    t0 = time.perf_counter()
    for _ in range(reps):
        orc.sha3_batch(buf, off, 256, threads=threads, lean=lean)
    dt = time.perf_counter() - t0
    return n * reps * MSG_LEN / dt / 1e9, n * reps


def cpu_sha3_baseline(budget_s: float, threads: int = 0):
    """The CPU baselines BASELINE.md 2 names, on this box's host cores, SHA3-256 over 64-byte messages:
      value / B-ref-parallel  the C restatement of Message::compute_sha3_hash (oracle/ref_cpu.c: message copy + pad +
                              the wasted post-squeeze permutation, like the Rust code) under an OpenMP loop over
                              messages (= a rayon par_iter wrapper), all host threads
      serial_1core            the same code looped one message at a time on ONE core -- what the reference does today
                              (src/sha3/hashable.rs:19-21 has no rayon)
      lean_1core / lean_parallel  the restatement without the copy and the wasted permutation
      openssl_1core           hashlib.sha3_256 (OpenSSL), one core, Python call overhead included
    """
    import hashlib

    import numpy as np

    from oracle import cpu

    orc = cpu.get(native=True)
    cores = host_threads() if threads <= 0 else threads
    par, n_par = _time_sha3(orc, 1 << 18, cores, 0, budget_s)
    ser, n_ser = _time_sha3(orc, 1 << 15, 1, 0, budget_s / 2)
    lean1, _ = _time_sha3(orc, 1 << 15, 1, 1, budget_s / 2)
    leanp, _ = _time_sha3(orc, 1 << 18, cores, 1, budget_s / 2)
    rng = np.random.default_rng(1)
    msgs = [rng.integers(0, 256, size=MSG_LEN, dtype=np.uint8).tobytes() for _ in range(1 << 15)]
    t0 = time.perf_counter()
    for m in msgs:
        hashlib.sha3_256(m).digest()
    ossl = len(msgs) * MSG_LEN / (time.perf_counter() - t0) / 1e9
    return {
        "value": par,
        "unit": "GB/s",
        "cores": cores,
        "kind": "port",
        "sample": f"{n_par} messages x {MSG_LEN} B, SHA3-256, oracle/ref_cpu.c (C restatement of the reference's "
                  f"Rust path incl. its message copy and extra permutation), gcc -O3 -march=native, {cores} threads "
                  f"(B-ref-parallel of BASELINE.md 2)",
        "msgs_per_s": par * 1e9 / MSG_LEN,
        "legs": {
            "serial_1core": {"value": ser, "unit": "GB/s", "cores": 1, "sample": f"{n_ser} messages, same code, one core: "
                             "what Message::compute_sha3_hash looped does today (no rayon on this path)"},
            "lean_1core": {"value": lean1, "unit": "GB/s", "cores": 1,
                           "sample": "restatement without the message copy and the wasted post-squeeze permutation"},
            "lean_parallel": {"value": leanp, "unit": "GB/s", "cores": cores, "sample": "lean variant, all host threads"},
            "openssl_1core": {"value": ossl, "unit": "GB/s", "cores": 1,
                              "sample": f"hashlib.sha3_256 over {len(msgs)} x {MSG_LEN} B (OpenSSL; Python call overhead included)"},
        },
    }


def cpu_ed448_baseline(budget_s: float, threads: int = 0):
    """The Ed448 half of the metric on the host: KeyPair::new-style [s]G (the reference multiplies the generator with
    its generic variable-base routine, ecc/keypair.rs:44), sign and verify, through the C restatement on `threads`
    host threads (0 = all) and on one core (what the reference does today), plus OpenSSL Ed448 (`cryptography`) on one
    core as an outside yardstick (a different signature protocol).  Bounded samples sized from a calibration run."""
    import numpy as np

    from oracle import cpu

    orc = cpu.get(native=True)
    cores = host_threads() if threads <= 0 else threads
    rng = np.random.default_rng(3)

    def rate(fn, n_cal, make, budget):
        args = make(n_cal)
        fn(*args)
        t0 = time.perf_counter()
        fn(*args)
        r = n_cal / (time.perf_counter() - t0)
        n = int(max(n_cal, min(1 << 16, r * budget)))
        args = make(n)
        t0 = time.perf_counter()
        fn(*args)
        return n / (time.perf_counter() - t0), n

    def mk_sc(n):
        return (rng.integers(0, 256, size=n * 56, dtype=np.uint8),)

    def mk_sign(n):
        pw = rng.integers(0, 256, size=n * 32, dtype=np.uint8)
        msg = rng.integers(0, 256, size=n * 256, dtype=np.uint8)
        return pw, np.arange(n + 1, dtype=np.uint64) * 32, msg, np.arange(n + 1, dtype=np.uint64) * 256

    def measure(t, budget):
        fb, n_fb = rate(lambda sc: orc.fixed_base_batch(sc, threads=t), 64 * t, mk_sc, budget)
        sg, n_sg = rate(lambda pw, po, m, mo: orc.sign_batch(pw, po, m, mo, 512, threads=t), 64 * t, mk_sign, budget)
        pw, po, m, mo = mk_sign(min(n_sg, 2048))
        pub = orc.keygen_batch(pw, po, 512, threads=t)
        h, z = orc.sign_batch(pw, po, m, mo, 512, threads=t)
        t0 = time.perf_counter()
        orc.verify_batch(pub, m, mo, h, z, 512, threads=t)
        vf = (len(po) - 1) / (time.perf_counter() - t0)
        return {"scalar_mults_per_s": fb, "signs_per_s": sg, "verifies_per_s": vf, "cores": t,
                "sample": f"{n_fb} generator multiplications, {n_sg} signatures, {len(po) - 1} verifications"}

    par = measure(cores, budget_s)
    out = {**par, "unit": "1/s", "kind": "port",
           "sample": par["sample"] + f" (32-byte passwords, 256-byte messages, D512), oracle/ref_cpu.c (64-bit limbs, u128 "
                                     f"products, signed radix-16 window like the crate), gcc -O3 -march=native, {cores} threads",
           "legs": {"serial_1core": measure(1, budget_s / 2)}}
    try:  # B-openssl: outside yardstick, one core
        from cryptography.hazmat.primitives.asymmetric.ed448 import Ed448PrivateKey

        n = 200
        msg = bytes(256)
        t0 = time.perf_counter()
        keys = [Ed448PrivateKey.generate() for _ in range(n)]
        pubs = [k.public_key() for k in keys]
        t_k = time.perf_counter() - t0
        t0 = time.perf_counter()
        sigs = [k.sign(msg) for k in keys]
        t_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        for p_, s_ in zip(pubs, sigs):
            p_.verify(s_, msg)
        t_v = time.perf_counter() - t0
        out["legs"]["openssl_1core"] = {"scalar_mults_per_s": n / t_k, "signs_per_s": n / t_s, "verifies_per_s": n / t_v,
                                        "cores": 1, "sample": f"{n} x OpenSSL Ed448 (RFC 8032 EdDSA, not the reference's "
                                                              "Schnorr variant) keygen / sign 256 B / verify via `cryptography`"}
    except Exception as e:  # pragma: no cover
        out["legs"]["openssl_1core"] = {"unavailable": repr(e)}
    return out


def run_reference(args, rank: int):
    """--impl reference: the reference's own CPU implementation of the path on the host cores.  The Rust
    reference cannot be built in this image (no rustc/cargo), so this is the oracle port.  The same program at every
    N: rank 0 alone runs it, on every host thread the process may use (explicit thread count -- torchrun's
    OMP_NUM_THREADS=1 does not apply)."""
    if rank != 0:
        return
    import numpy as np

    from oracle import cpu

    orc = cpu.get(native=True)
    cores = host_threads()
    rng = np.random.default_rng(1)
    n_cal = 1 << 16
    buf = rng.integers(0, 256, size=n_cal * MSG_LEN, dtype=np.uint8)
    off = np.arange(n_cal + 1, dtype=np.uint64) * MSG_LEN
    orc.sha3_batch(buf, off, 256, threads=cores)
    t0 = time.perf_counter()
    orc.sha3_batch(buf, off, 256, threads=cores)
    rate = n_cal / (time.perf_counter() - t0)
    total_budget_s = 90.0
    n = int(min(N_MSGS, max(4096, rate * total_budget_s / max(1, args.steps + args.warmup))))
    buf = rng.integers(0, 256, size=n * MSG_LEN, dtype=np.uint8)
    off = np.arange(n + 1, dtype=np.uint64) * MSG_LEN
    for _ in range(args.warmup):
        orc.sha3_batch(buf, off, 256, threads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.sha3_batch(buf, off, 256, threads=cores)
    dt = time.perf_counter() - t0
    gbps = n * args.steps * MSG_LEN / dt / 1e9
    sample = (f"each step = {n} of the {N_MSGS} messages x {MSG_LEN} B (bounded sample), oracle/ref_cpu.c restatement of "
              f"Message::compute_sha3_hash looped, gcc -O3 -march=native, {cores} threads")
    line = {
        "impl": "reference", "metric": "sha3_256_GBps", "value": gbps, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(), "sample_msgs_per_step": n,
        "cpu_baseline": {"value": gbps, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": gbps, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extra": {"ed448_cpu": cpu_ed448_baseline(budget_s=1.0, threads=cores)},
    }
    emit_json_line(line)


# ------------------------------------------------------------------------------------------------------
def live_peaks():
    """Integer-pipe peaks measured now on this GPU by the in-tree microbenchmark (csrc/peaks.cu)."""
    exe = os.path.join(ROOT, "capycrypt_b200", "_lib", "peaks")
    try:
        r = subprocess.run([exe, "600"], capture_output=True, text=True, timeout=120)
        d = json.loads(r.stdout.strip().splitlines()[-1])
        return {"lop3": d["lop3"]["thread_ops_per_s"], "imad_wide": d["imad_wide"]["thread_ops_per_s"],
                "source": "measured live by capycrypt_b200/_lib/peaks (csrc/peaks.cu)"}
    except Exception as e:
        return {**PEAK_FALLBACK, "source": f"profiles/r01_peaks_int_pipes.json (live run failed: {e!r})"}


def bind_to_gpu_numa_node(local: int):
    """Pins this rank's process to the CPUs NVML reports as closest to its GPU, so that the pinned host buffers of the
    end-to-end leg are first-touched on that NUMA node (one process per GPU: without this all ranks' buffers tend to land
    on one socket and the host side of PCIe becomes the bottleneck at N > 1).  Harness plumbing, not part of the engine."""
    try:
        import pynvml as nv

        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = nv.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1 and 64 * w + b < ncpu}
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return {"cpus": len(allowed), "first": min(allowed), "last": max(allowed)}
    except Exception as e:  # pragma: no cover
        return {"error": repr(e)}
    return None


_REAL_STDOUT = None


def keep_stdout_for_the_json_line():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout when
    NCCL_DEBUG is set), so file descriptor 1 is pointed at stderr for the whole run and the line goes to a saved copy
    of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json_line(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def dump_outputs(path: str, digests):
    """Saves what the timed path returned in its last step, so that two builds can be compared output for output: the
    SHA3-256 digests of DUMP_ROWS messages drawn with DUMP_SEED, in message order, one float32 per digest byte."""
    import numpy as np
    import torch

    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(N_MSGS, DUMP_ROWS, replace=False))
    sample = digests.view(N_MSGS, DIGEST)[torch.from_numpy(rows).to(digests.device)].cpu().numpy()
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "sha3_256_digests.npy"), sample.astype(np.float32))


def main():
    keep_stdout_for_the_json_line()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the Ed448 / KMAC side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write a seeded sample of rank 0's last-step digests to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3)
    rank, world, local = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch

    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)  # before any host buffer is allocated (first touch decides the NUMA node)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    from capycrypt_b200 import Engine

    eng = Engine()  # one ctx on this rank's GPU
    dev = torch.device("cuda", local)
    g = torch.Generator(device=dev)
    g.manual_seed(1 + rank)
    ins = [torch.randint(0, 256, (N_MSGS * MSG_LEN,), dtype=torch.uint8, device=dev, generator=g) for _ in range(N_ROT)]
    outs = [torch.zeros(N_MSGS * DIGEST, dtype=torch.uint8, device=dev) for _ in range(N_ROT)]

    def step(i):
        eng.sha3_fixed_dev(ins[i % N_ROT], MSG_LEN, MSG_LEN, N_MSGS, 256, outs[i % N_ROT])

    peaks = live_peaks() if rank == 0 else PEAK_FALLBACK
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    # sanity (not the oracle): SHA3-256 is FIPS-exact in the reference for every length
    import hashlib

    m0 = ins[0][:MSG_LEN].cpu().numpy().tobytes()
    assert outs[0][:DIGEST].cpu().numpy().tobytes() == hashlib.sha3_256(m0).digest(), "digest mismatch"

    sampler = ClockSampler(local)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    if dist:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launch_count - launches0
    if dist:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = world * N_MSGS * MSG_LEN / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs[(args.steps - 1) % N_ROT])

    # ---- e2e: the same metric through the host-buffer C entry point (pinned host memory, H2D + D2H inside) ----
    k_e2e = max(5, min(args.steps, 100))
    h_in = eng.pinned(N_MSGS * MSG_LEN)
    h_out = eng.pinned(N_MSGS * DIGEST)
    h_in[:] = ins[0].cpu().numpy()
    h_out2d = h_out.reshape(N_MSGS, DIGEST)
    for _ in range(3):
        eng.sha3_fixed(h_in, MSG_LEN, MSG_LEN, N_MSGS, 256, out=h_out2d)
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(k_e2e):
        eng.sha3_fixed(h_in, MSG_LEN, MSG_LEN, N_MSGS, 256, out=h_out2d)
    e2e_s = time.perf_counter() - t0
    if dist:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    assert h_out[:DIGEST].tobytes() == hashlib.sha3_256(m0).digest()
    # the same call from ordinary (pageable) memory -- what a caller gets that hands over a Vec / numpy array instead of
    # packing into a capy_host_alloc buffer: the driver stages such copies through its own pinned buffers
    p_in, p_out = np.array(h_in), np.zeros((N_MSGS, DIGEST), np.uint8)
    eng.sha3_fixed(p_in, MSG_LEN, MSG_LEN, N_MSGS, 256, out=p_out)
    t0 = time.perf_counter()
    for _ in range(5):
        eng.sha3_fixed(p_in, MSG_LEN, MSG_LEN, N_MSGS, 256, out=p_out)
    pageable_s = (time.perf_counter() - t0) / 5
    assert np.array_equal(p_out, h_out2d)
    del p_in, p_out
    # the denominator of the end-to-end number: the same bytes, the same pinned buffers, every rank at the same time,
    # plain cudaMemcpyAsync in both directions and no kernel (capy_copy_probe)
    if dist:
        dist.barrier()
    link_ms = eng.copy_probe(h_in, h_out, reps=10)
    if dist:
        t = torch.tensor([link_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        link_ms = float(t.item())
    e2e_val = world * N_MSGS * MSG_LEN * k_e2e / e2e_s / 1e9
    link_ceiling = world * N_MSGS * MSG_LEN / (link_ms * 1e-3) / 1e9
    e2e = {"value": e2e_val, "unit": "GB/s",
           "h2d_bytes_per_step": N_MSGS * MSG_LEN, "d2h_bytes_per_step": N_MSGS * DIGEST, "steps": k_e2e,
           "ms_per_step": e2e_s / k_e2e * 1e3,
           "api": "capy_sha3_batch_fixed (host buffers from capy_host_alloc, chunked H2D/kernel/D2H on 3 streams)",
           "link_ceiling_GBps": link_ceiling, "link_ms_per_step": link_ms, "frac_of_link": e2e_val / link_ceiling,
           "link_probe": "capy_copy_probe: 64 MiB H2D + 32 MiB D2H per rank from the same pinned buffers, both directions "
                         "overlapped, all ranks concurrently, no kernel (max over ranks)",
           "host_numa_binding": numa,
           "pageable_buffers_GBps_this_rank": N_MSGS * MSG_LEN / pageable_s / 1e9}

    # ---- roofline of the dominant kernel (sha3_short_kernel<17, 8>: one launch per step) ----
    ops = N_MSGS * OPS_PER_PERM
    achieved = ops / (ms_per_step * 1e-3) * (1 if world == 1 else 1)  # per GPU
    hbm_bytes = N_MSGS * (MSG_LEN + DIGEST)
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        hbm_src = "MEASURED_PEAKS.json"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("sha3_short_kernel<17, 8>")
    except Exception:
        pass
    roofline = {
        "bound": "int_alu", "kernel": "sha3_short_kernel<17, 8>", "achieved": achieved / 1e12, "peak": peaks["lop3"] / 1e12,
        "unit": "Tint32op/s", "frac": achieved / peaks["lop3"], "traffic": traffic,
        "peak_source": peaks.get("source", "profiles/r01_peaks_int_pipes.json"),
        "algorithmic": f"{OPS_PER_PERM} int32 LOP3/SHF per Keccak-f[1600] x 1 permutation x {N_MSGS} messages per launch",
        "hbm": {"achieved": hbm_bytes / (ms_per_step * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": hbm_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src,
                "algorithmic": "64 B in + 32 B out per message"},
        "note": "the path is integer-ALU bound (BASELINE.md 4): the binding roofline is the measured LOP3/SHF pipe peak, "
                "the HBM fraction is reported beside it",
    }

    line = {
        "metric": "sha3_256_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
        "msgs_per_s": world * N_MSGS / (ms_per_step * 1e-3),
    }

    if not args.no_extras:
        line["extra"] = extras(eng, dev, peaks, world, dist, rank)
    if rank == 0 and world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_sha3_baseline(budget_s=1.5)
        line["cpu_baseline"]["ed448"] = cpu_ed448_baseline(budget_s=1.0)
    elif rank == 0:
        line["cpu_baseline"] = None
    eng.close()
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit_json_line(line)


def lpt_shards(lens, world):
    """Longest-processing-time-first assignment of messages to ranks (SURVEY 8e): every message goes, longest first, to
    the rank with the least work so far.  Returns a list of index arrays, one per rank."""
    import heapq

    import numpy as np

    order = np.argsort(-lens, kind="stable")
    heap = [(0, r) for r in range(world)]
    shards = [[] for _ in range(world)]
    for i in order:
        load, r = heapq.heappop(heap)
        shards[r].append(int(i))
        heapq.heappush(heap, (load + int(lens[i]) // 72 + 2, r))
    return [np.sort(np.array(sh, dtype=np.int64)) for sh in shards]


def _oracle():
    """The checker (oracle/ref_cpu.c) for the sampled parity checks of the extras -- outside every timed region."""
    from oracle import cpu

    return cpu.get()


def extras(eng, dev, peaks, world, dist, rank):
    """Side measurements for the other BASELINE.json configs (device-resident, CUDA events, max over ranks), each
    followed -- outside its timed region -- by a check of a seeded sample of its results against the C oracle, and
    host-buffer (e2e) figures for cfg 2, 4 and 5 through the blocking C entry points with pinned buffers."""
    import time as _t

    import numpy as np
    import torch

    orc = _oracle()
    eng.set_plan_cache(True)  # ragged _dev calls that pass the same offsets array again launch without a host round trip

    def timed(fn, steps, warmup=2):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if dist:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed_host(fn, steps, warmup=1):
        for _ in range(warmup):
            fn()
        if dist:
            dist.barrier()
        t0 = _t.perf_counter()
        for _ in range(steps):
            fn()
        dt = (_t.perf_counter() - t0) / steps
        if dist:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt

    def rows(t, n, w, idx):  # sample rows of a device tensor as one packed numpy array
        return t.view(n, w)[torch.from_numpy(idx).to(dev)].cpu().numpy().reshape(-1)

    g = torch.Generator(device=dev)
    g.manual_seed(100 + rank)
    rnd = lambda n: torch.randint(0, 256, (n,), dtype=torch.uint8, device=dev, generator=g)
    rs_np = np.random.default_rng(1000 + rank)
    out = {}
    NS = 256  # oracle sample per check

    # ---- cfg 2: KMACXOF256 (D512) over 2^16 x 4 KB messages, 32-byte keys, 512-bit output --------------------------
    n2, mlen = 1 << 16, 4096
    data, keys = rnd(n2 * mlen), rnd(n2 * 32)
    o = torch.zeros(n2 * 64, dtype=torch.uint8, device=dev)
    custom = b"My Tagged Application"
    ms = timed(lambda: eng.kmac_xof_fixed_dev(keys, 32, 32, data, mlen, mlen, n2, 512, custom, 512, o), 10)
    idx2 = np.sort(rs_np.choice(n2, size=NS, replace=False))
    s_data, s_keys = rows(data, n2, mlen, idx2), rows(keys, n2, 32, idx2)
    s_off, s_koff = np.arange(NS + 1, dtype=np.uint64) * mlen, np.arange(NS + 1, dtype=np.uint64) * 32
    assert np.array_equal(rows(o, n2, 64, idx2).reshape(NS, 64),
                          orc.kmac_xof_batch(s_keys, s_koff, s_data, s_off, 512, custom, 512)), "cfg 2: KMACXOF256 != oracle"
    perms = 32  # 33 absorbed blocks, the constant prefix block is cached
    out["kmac256_2^16x4KB"] = {
        "GBps": world * n2 * mlen / (ms * 1e-3) / 1e9, "ms_per_step": ms,
        "frac_int_alu": n2 * perms * OPS_PER_PERM / (ms * 1e-3) / peaks["lop3"], "perms_per_msg": perms,
        "oracle_sample": NS,
        "launch": "sponge_chain_kernel: 2 048 warps on 592 schedulers = 3.46 each, so the chains are cut in two dependent jobs "
                  "of one launch (6.92 warps per scheduler); CAPY_NO_CHAIN_SPLIT=1 gives the uncut launch"}

    # cfg 2, variable-length squeeze: cSHAKE256 and KMACXOF256 with a 4 096-byte output per message (the keystream shape of
    # sha3/encryptable.rs:41), and FIPS 202 SHAKE256 (no reference counterpart) with a 64-byte output
    off2 = torch.arange(n2 + 1, dtype=torch.int64, device=dev) * mlen
    koff2 = torch.arange(n2 + 1, dtype=torch.int64, device=dev) * 32
    big = torch.zeros(n2 * 4096, dtype=torch.uint8, device=dev)
    ms_c = timed(lambda: eng.cshake_dev(data, off2, 8 * 4096, b"", b"Email Signature", 512, big), 5)
    assert np.array_equal(rows(big, n2, 4096, idx2[:32]).reshape(32, 4096),
                          orc.cshake_batch(s_data[: 32 * mlen], s_off[:33], 8 * 4096, b"", b"Email Signature", 512)), "cSHAKE256 != oracle"
    ms_k = timed(lambda: eng.kmac_xof_dev(keys, koff2, data, off2, 8 * 4096, custom, 512, big), 5)
    assert np.array_equal(rows(big, n2, 4096, idx2[:32]).reshape(32, 4096),
                          orc.kmac_xof_batch(s_keys[: 32 * 32], s_koff[:33], s_data[: 32 * mlen], s_off[:33], 8 * 4096, custom, 512)), \
        "KMACXOF256 (4 KB out) != oracle"
    ms_s = timed(lambda: eng.fips_shake_dev(data, off2, 256, 64, o), 5)
    import hashlib

    m0 = data[:mlen].cpu().numpy().tobytes()
    assert o[:64].cpu().numpy().tobytes() == hashlib.shake_256(m0).digest(64), "FIPS SHAKE256 != hashlib"
    sq = (4096 + 135) // 136 - 1  # extra permutations of a 4 096-byte squeeze at rate 136
    out["cfg2_variable_squeeze_2^16x4KB"] = {
        "cshake256_out4096B_ms": ms_c, "cshake256_out4096B_GBps_in_plus_out": world * n2 * (mlen + 4096) / (ms_c * 1e-3) / 1e9,
        "cshake256_frac_int_alu": n2 * (31 + sq) * OPS_PER_PERM / (ms_c * 1e-3) / peaks["lop3"],
        "kmacxof256_out4096B_ms": ms_k, "kmacxof256_frac_int_alu": n2 * (32 + sq) * OPS_PER_PERM / (ms_k * 1e-3) / peaks["lop3"],
        "fips_shake256_out64B_ms": ms_s, "fips_shake256_GBps": world * n2 * mlen / (ms_s * 1e-3) / 1e9,
        "fips_shake256_frac_int_alu": n2 * 31 * OPS_PER_PERM / (ms_s * 1e-3) / peaks["lop3"]}
    del big

    # cfg 2 end to end: host buffers (pinned, capy_host_alloc) through capy_kmac_xof_batch, H2D of keys + messages +
    # offsets and D2H of the tags inside the timed region
    h_data, h_keys = eng.pinned(n2 * mlen), eng.pinned(n2 * 32)
    h_data[:] = data.cpu().numpy()
    h_keys[:] = keys.cpu().numpy()
    np_off, np_koff = np.arange(n2 + 1, dtype=np.uint64) * mlen, np.arange(n2 + 1, dtype=np.uint64) * 32
    res = {}
    h_tags = eng.pinned(n2 * 64).reshape(n2, 64)  # results land in pinned memory too (a pageable target halves the D2H rate)
    dt = timed_host(lambda: res.__setitem__("t", eng.kmac_xof(h_keys, np_koff, h_data, np_off, 512, custom, 512, out=h_tags)), 3)
    assert np.array_equal(res["t"][idx2], orc.kmac_xof_batch(s_keys, s_koff, s_data, s_off, 512, custom, 512)), "cfg 2 e2e != oracle"
    out["kmac256_2^16x4KB"]["e2e"] = {
        "GBps": world * n2 * mlen / dt / 1e9, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": n2 * (mlen + 32 + 16),
        "d2h_bytes_per_step": n2 * 64, "api": "capy_kmac_xof_batch (pinned host buffers from capy_host_alloc)"}
    del h_data, h_keys

    # ---- cfg 5: mixed-size SHA3-512, lengths log-uniform in [64 B, 1 MiB], 16 GiB in total (strong scaling: the 16 GiB
    # are split over the ranks longest-first, LPT); one launch, three tiers ------------------------------------------
    rs = np.random.default_rng(5)
    total = 16 << 30
    lens, acc = [], 0
    while acc < total:
        c = np.exp(rs.uniform(np.log(64), np.log(1 << 20), size=8192)).astype(np.int64)
        lens.append(c)
        acc += int(c.sum())
    lens_all = np.concatenate(lens)
    lens_all = lens_all[: int(np.searchsorted(np.cumsum(lens_all), total)) + 1]
    lens = lens_all[lpt_shards(lens_all, world)[rank]] if world > 1 else lens_all
    off5 = np.zeros(len(lens) + 1, np.int64)
    off5[1:] = np.cumsum(lens)
    nbytes5 = int(off5[-1])
    d5 = torch.empty(nbytes5 + 8, dtype=torch.uint8, device=dev)
    d5.random_(0, 256, generator=g)
    t_off5 = torch.from_numpy(off5).to(dev)
    o5 = torch.zeros(len(lens) * 64, dtype=torch.uint8, device=dev)
    ms = timed(lambda: eng.sha3_dev(d5, t_off5, 512, o5), 2, 1)
    # sampled oracle check: every quirk length in a window, the longest (fast-tier) messages, random others
    quirk = np.nonzero((lens % 72 == 71) | (lens % 136 == 135))[0][:64]
    pick = np.unique(np.concatenate([quirk, np.argsort(lens)[-8:], rs_np.choice(len(lens), size=NS, replace=False)]))
    d5_np = [d5[int(off5[i]):int(off5[i + 1])].cpu().numpy() for i in pick]
    s5_off = np.zeros(len(pick) + 1, np.uint64)
    s5_off[1:] = np.cumsum([len(x) for x in d5_np])
    assert np.array_equal(o5.view(len(lens), 64)[torch.from_numpy(pick).to(dev)].cpu().numpy(),
                          orc.sha3_batch(np.concatenate(d5_np), s5_off, 512, threads=0)), "cfg 5: SHA3-512 != oracle"
    del d5_np
    # A/B: the same batch with one thread per message everywhere (CAPY_FLAG_NO_PAIR = 2)
    ms_solo = timed(lambda: eng._check(eng.lib.capy_sha3_batch_dev(eng._ctx, 0, eng._stream(), 512, d5.data_ptr(),
                                                                   t_off5.data_ptr(), len(lens), o5.data_ptr(), 2)), 1, 1)
    perms5 = int(((lens + 1 + 71) // 72).sum())
    longest = int((lens.max() + 1 + 71) // 72)
    tot_bytes = torch.tensor([float(nbytes5)], device=dev, dtype=torch.float64)
    tot_perms = torch.tensor([float(perms5)], device=dev, dtype=torch.float64)
    max_chain = torch.tensor([float(longest)], device=dev, dtype=torch.float64)
    max_perms = torch.tensor([float(perms5)], device=dev, dtype=torch.float64)
    if dist:
        dist.all_reduce(tot_bytes)
        dist.all_reduce(tot_perms)
        dist.all_reduce(max_chain, op=dist.ReduceOp.MAX)
        dist.all_reduce(max_perms, op=dist.ReduceOp.MAX)
    chain_floor_ms = float(max_chain.item()) * WARP_TIER_US_PER_PERM * 1e-3
    work_floor_ms = float(max_perms.item()) * OPS_PER_PERM / peaks["lop3"] * 1e3
    floor_ms = max(chain_floor_ms, work_floor_ms)
    out["sha3_512_mixed_16GiB"] = {
        "GBps": float(tot_bytes.item()) / (ms * 1e-3) / 1e9, "ms_per_step": ms, "msgs_this_rank": int(len(lens)),
        "frac_int_alu": float(tot_perms.item()) / world * OPS_PER_PERM / (ms * 1e-3) / peaks["lop3"],
        "scaling": "strong", "sharding": "LPT over all messages by permutation count (longest first to the least loaded rank)",
        "longest_chain_perms": longest, "chain_floor_ms": chain_floor_ms, "work_floor_ms": work_floor_ms,
        "frac_of_floor": floor_ms / ms, "ms_one_thread_per_message": ms_solo, "oracle_sample": int(len(pick)),
        "note": "a sponge is sequential per message: the step cannot be shorter than the longest message's chain at the "
                "fastest tier (1 MiB = 14 564 permutations x 2.04 us with a whole warp per message = chain_floor_ms) nor than "
                "the rank's permutations at the ALU peak (work_floor_ms); frac_of_floor = max of the two / measured"}
    del d5, o5, t_off5

    # cfg 5 end to end: a 2 GiB shard (the share of one rank of an 8-GPU run) from pinned host memory through capy_sha3_batch
    lens_e = lens_all[lpt_shards(lens_all, 8)[rank % 8]]
    off_e = np.zeros(len(lens_e) + 1, np.uint64)
    off_e[1:] = np.cumsum(lens_e)
    nb_e = int(off_e[-1])
    h5 = eng.pinned(nb_e)
    blk = rs_np.integers(0, 256, size=64 << 20, dtype=np.uint8)
    for p0 in range(0, nb_e, len(blk)):
        h5[p0:p0 + len(blk)] = blk[: min(len(blk), nb_e - p0)]
    h5_out = eng.pinned(len(lens_e) * 64).reshape(len(lens_e), 64)
    dt = timed_host(lambda: res.__setitem__("d", eng.sha3(h5, off_e, 512, out=h5_out)), 2)
    pick = np.unique(np.concatenate([np.argsort(lens_e)[-4:], rs_np.choice(len(lens_e), size=NS, replace=False)]))
    sm = [h5[int(off_e[i]):int(off_e[i + 1])] for i in pick]
    s_o = np.zeros(len(pick) + 1, np.uint64)
    s_o[1:] = np.cumsum([len(x) for x in sm])
    assert np.array_equal(res["d"][pick], orc.sha3_batch(np.concatenate(sm), s_o, 512, threads=0)), "cfg 5 e2e != oracle"
    out["sha3_512_mixed_16GiB"]["e2e_2GiB_shard"] = {
        "GBps": world * nb_e / dt / 1e9, "ms_per_step": dt * 1e3, "bytes": nb_e, "msgs": int(len(lens_e)),
        "h2d_bytes_per_step": nb_e + 8 * (len(lens_e) + 1), "d2h_bytes_per_step": 64 * len(lens_e),
        "api": "capy_sha3_batch (pinned host buffers from capy_host_alloc; one rank's LPT shard of the 8-GPU run)"}
    del h5, sm

    # ---- cfg 3: Ed448 fixed-base [s]G for 2^20 scalars ------------------------------------------------------------
    n3 = 1 << 20
    sc = rnd(n3 * 56)
    pts = torch.zeros(n3 * 112, dtype=torch.uint8, device=dev)
    ms = timed(lambda: eng.ed448_fixed_base_dev(sc, n3, pts), 3, 1)
    idx3 = np.sort(rs_np.choice(n3, size=NS, replace=False))
    assert np.array_equal(rows(pts, n3, 112, idx3).reshape(NS, 112), orc.fixed_base_batch(rows(sc, n3, 56, idx3), threads=0)), \
        "cfg 3: [s]G != oracle"
    rate = n3 / (ms * 1e-3)
    out["ed448_fixed_base_2^20"] = {
        "scalar_mults_per_s": world * rate, "ms_per_step": ms, "frac_imad_wide": rate * MAC_FIXED / peaks["imad_wide"],
        "canonical_macs": MAC_FIXED, "executed_imad_wide": MAC_EXEC_FIXED,
        "frac_imad_wide_executed": rate * MAC_EXEC_FIXED / peaks["imad_wide"], "constant_time_lookup": True, "oracle_sample": NS,
        "note": "frac_imad_wide = canonical-budget MACs/s / IMAD.WIDE peak (comparable across designs; can exceed the pipe's "
                "real utilisation because the comb on the isogenous curve executes fewer MACs); frac_imad_wide_executed = "
                "IMAD.WIDE instructions actually issued / peak"}

    # variable base for 2^18 (scalar, point) pairs
    n4 = 1 << 18
    o4 = torch.zeros(n4 * 112, dtype=torch.uint8, device=dev)
    ms = timed(lambda: eng.ed448_var_base_dev(sc, pts, n4, o4), 2, 1)
    idx4 = np.sort(rs_np.choice(n4, size=NS, replace=False))
    rc_o, want = orc.var_base_batch(rows(sc, n3, 56, idx4), rows(pts, n3, 112, idx4), threads=0)
    assert rc_o == 0 and np.array_equal(rows(o4, n4, 112, idx4).reshape(NS, 112), want), "[k]P != oracle"
    rate = n4 / (ms * 1e-3)
    out["ed448_var_base_2^18"] = {
        "scalar_mults_per_s": world * rate, "ms_per_step": ms, "frac_imad_wide": rate * MAC_VAR / peaks["imad_wide"],
        "canonical_macs": MAC_VAR, "executed_imad_wide": MAC_EXEC_VAR,
        "frac_imad_wide_executed": rate * MAC_EXEC_VAR / peaks["imad_wide"], "constant_time_lookup": True, "oracle_sample": NS}

    # ---- cfg 4: Schnorr sign + verify, 2^18 x (32-byte password, 256-byte message), D512 ---------------------------
    pw, msg = rnd(n4 * 32), rnd(n4 * 256)
    pw_off = torch.arange(n4 + 1, dtype=torch.int64, device=dev) * 32
    msg_off = torch.arange(n4 + 1, dtype=torch.int64, device=dev) * 256
    h = torch.zeros(n4 * 56, dtype=torch.uint8, device=dev)
    z = torch.zeros(n4 * 56, dtype=torch.uint8, device=dev)
    pub = torch.zeros(n4 * 112, dtype=torch.uint8, device=dev)
    ok = torch.zeros(n4, dtype=torch.uint8, device=dev)
    ms_k = timed(lambda: eng.ed448_keygen_dev(pw, pw_off, 512, pub), 2, 1)
    ms_s = timed(lambda: eng.ed448_sign_dev(pw, pw_off, msg, msg_off, 512, h, z), 2, 1)
    ms_v = timed(lambda: eng.ed448_verify_dev(pub, msg, msg_off, h, z, 512, ok), 2, 1)
    s_pw, s_msg = rows(pw, n4, 32, idx4), rows(msg, n4, 256, idx4)
    s_po, s_mo = np.arange(NS + 1, dtype=np.uint64) * 32, np.arange(NS + 1, dtype=np.uint64) * 256
    h_ref, z_ref = orc.sign_batch(s_pw, s_po, s_msg, s_mo, 512, threads=0)
    assert np.array_equal(rows(pub, n4, 112, idx4).reshape(NS, 112), orc.keygen_batch(s_pw, s_po, 512, threads=0)), "cfg 4: keygen != oracle"
    assert np.array_equal(rows(h, n4, 56, idx4).reshape(NS, 56), h_ref) and np.array_equal(rows(z, n4, 56, idx4).reshape(NS, 56), z_ref), \
        "cfg 4: signatures != oracle"
    assert bool(ok.all().item()), "cfg 4: the engine rejected its own signatures"
    assert orc.verify_batch(rows(pub, n4, 112, idx4), s_msg, s_mo, h_ref.reshape(-1), z_ref.reshape(-1), 512, threads=0).all()
    out["ed448_schnorr_2^18x256B"] = {
        "keygens_per_s": world * n4 / (ms_k * 1e-3), "signs_per_s": world * n4 / (ms_s * 1e-3),
        "verifies_per_s": world * n4 / (ms_v * 1e-3), "ms_keygen": ms_k, "ms_sign": ms_s, "ms_verify": ms_v, "oracle_sample": NS}
    # cfg 4 end to end: pinned host buffers through capy_ed448_sign_batch / capy_ed448_verify_batch
    h_pw, h_msg = eng.pinned(n4 * 32), eng.pinned(n4 * 256)
    h_pw[:] = pw.cpu().numpy()
    h_msg[:] = msg.cpu().numpy()
    np_po, np_mo = np.arange(n4 + 1, dtype=np.uint64) * 32, np.arange(n4 + 1, dtype=np.uint64) * 256
    h_h, h_z, h_pub, h_ok = (eng.pinned(n4 * 56).reshape(n4, 56), eng.pinned(n4 * 56).reshape(n4, 56), eng.pinned(n4 * 112),
                             eng.pinned(n4))
    h_pub[:] = pub.cpu().numpy()
    dt_s = timed_host(lambda: res.__setitem__("s", eng.ed448_sign(h_pw, np_po, h_msg, np_mo, 512, h_out=h_h, z_out=h_z)), 2)
    dt_v = timed_host(lambda: res.__setitem__("v", eng.ed448_verify(h_pub, h_msg, np_mo, h_h, h_z, 512, ok_out=h_ok)), 2)
    assert res["v"][0] == 0 and res["v"][1].all() and np.array_equal(h_h[idx4], h_ref) and np.array_equal(h_z[idx4], z_ref), "cfg 4 e2e"
    out["ed448_schnorr_2^18x256B"]["e2e"] = {
        "signs_per_s": world * n4 / dt_s, "verifies_per_s": world * n4 / dt_v, "ms_sign": dt_s * 1e3, "ms_verify": dt_v * 1e3,
        "h2d_bytes_per_sign": 32 + 256 + 16, "d2h_bytes_per_sign": 112, "h2d_bytes_per_verify": 112 + 256 + 8 + 112,
        "d2h_bytes_per_verify": 1, "api": "capy_ed448_sign_batch / capy_ed448_verify_batch (inputs and results in pinned host buffers from capy_host_alloc)"}
    del h_pw, h_msg
    # the other message sizes SURVEY 8(d) asks for (64 B and 4 KB) and cfg 3's password variant (2^20 x 32-byte passwords)
    for mlen4 in (64, 4096):
        msg_b = rnd(n4 * mlen4)
        off_b = torch.arange(n4 + 1, dtype=torch.int64, device=dev) * mlen4
        ms_s2 = timed(lambda: eng.ed448_sign_dev(pw, pw_off, msg_b, off_b, 512, h, z), 2, 1)
        ms_v2 = timed(lambda: eng.ed448_verify_dev(pub, msg_b, off_b, h, z, 512, ok), 2, 1)
        assert bool(ok.all().item())
        h_r2, z_r2 = orc.sign_batch(s_pw[: 32 * 32], s_po[:33], rows(msg_b, n4, mlen4, idx4[:32]), np.arange(33, dtype=np.uint64) * mlen4, 512, threads=0)
        assert np.array_equal(rows(h, n4, 56, idx4[:32]).reshape(32, 56), h_r2) and np.array_equal(rows(z, n4, 56, idx4[:32]).reshape(32, 56), z_r2)
        out[f"ed448_schnorr_2^18x{mlen4}B"] = {"signs_per_s": world * n4 / (ms_s2 * 1e-3), "verifies_per_s": world * n4 / (ms_v2 * 1e-3),
                                               "ms_sign": ms_s2, "ms_verify": ms_v2}
        del msg_b, off_b
    pw20 = rnd(n3 * 32)
    pw20_off = torch.arange(n3 + 1, dtype=torch.int64, device=dev) * 32
    pub20 = torch.zeros(n3 * 112, dtype=torch.uint8, device=dev)
    ms_k20 = timed(lambda: eng.ed448_keygen_dev(pw20, pw20_off, 512, pub20), 2, 1)
    assert np.array_equal(rows(pub20, n3, 112, idx3[:64]).reshape(64, 112),
                          orc.keygen_batch(rows(pw20, n3, 32, idx3[:64]), np.arange(65, dtype=np.uint64) * 32, 512, threads=0))
    out["ed448_keygen_2^20_passwords"] = {"keygens_per_s": world * n3 / (ms_k20 * 1e-3), "ms_per_step": ms_k20}
    del pw20, pw20_off, pub20
    eng.ed448_sign_dev(pw, pw_off, msg, msg_off, 512, h, z)  # h, z back to the 256-byte messages for what follows

    # ---- "next" rows N2 / N3 (SURVEY 8f): sponge AE over the cfg-2 shape (2^16 x 4 KB: the tag pass and the keystream pass
    # of the seal are one launch) and ECDHIES over 2^18 x 256 B, device-resident ------------------------------------
    from oracle import ref_sha3

    nonces = rnd(n2 * 512)
    pw2 = rnd(n2 * 32)
    pw2_off = torch.arange(n2 + 1, dtype=torch.int64, device=dev) * 32
    m_off = torch.arange(n2 + 1, dtype=torch.int64, device=dev) * mlen
    ct, pt = torch.empty_like(data), torch.empty_like(data)
    tag = torch.zeros(n2 * 64, dtype=torch.uint8, device=dev)
    ok2 = torch.zeros(n2, dtype=torch.uint8, device=dev)
    ms_e = timed(lambda: eng.sponge_encrypt_dev(pw2, pw2_off, n2 * 32, nonces, 512, data, m_off, 512, ct, tag), 5)
    ms_d = timed(lambda: eng.sponge_decrypt_dev(pw2, pw2_off, n2 * 32, nonces, 512, ct, m_off, tag, 512, pt, ok2), 5)
    assert bool(ok2.all().item()) and bool(torch.equal(pt, data)), "sponge AE round trip failed"
    for i in idx2[:4]:  # the Python restatement of sha3/encryptable.rs:29-45 (slow: a handful of messages)
        i = int(i)
        c_ref, t_ref = ref_sha3.sha3_encrypt(data[i * mlen:(i + 1) * mlen].cpu().numpy().tobytes(), pw2[i * 32:(i + 1) * 32].cpu().numpy().tobytes(),
                                             512, nonces[i * 512:(i + 1) * 512].cpu().numpy().tobytes())
        assert ct[i * mlen:(i + 1) * mlen].cpu().numpy().tobytes() == c_ref and tag[i * 64:(i + 1) * 64].cpu().numpy().tobytes() == t_ref, \
            "sha3_encrypt != oracle"
    ae_perms = 6 + 32 + 32  # key derivation (z || pw: 5 key blocks + 1) + tag pass + keystream (2 absorb + 30 squeeze); prefix cached
    out["sha3_encrypt_2^16x4KB"] = {
        "encrypt_GBps": world * n2 * mlen / (ms_e * 1e-3) / 1e9, "decrypt_GBps": world * n2 * mlen / (ms_d * 1e-3) / 1e9,
        "ms_encrypt": ms_e, "ms_decrypt": ms_d,
        "frac_int_alu_encrypt": n2 * ae_perms * OPS_PER_PERM / (ms_e * 1e-3) / peaks["lop3"],
        "frac_int_alu_decrypt": n2 * ae_perms * OPS_PER_PERM / (ms_d * 1e-3) / peaks["lop3"], "perms_per_msg": ae_perms}
    del ct, pt, nonces

    from oracle import ref_ed448

    n5 = n4  # 2^18 like cfg 4 (1 024 blocks of var_base_kernel = 6.92 per SM; 2^17 would be 3.46: a quarter wave idle)
    k_rand = rnd(n5 * 56)
    m5 = msg[: n5 * 256]
    m5_off = msg_off[: n5 + 1]
    ct5, pt5 = torch.empty_like(m5), torch.empty_like(m5)
    tag5 = torch.zeros(n5 * 56, dtype=torch.uint8, device=dev)
    zpt = torch.zeros(n5 * 112, dtype=torch.uint8, device=dev)
    ok5 = torch.zeros(n5, dtype=torch.uint8, device=dev)
    ms_e = timed(lambda: eng.ed448_key_encrypt_dev(pub, k_rand, m5, m5_off, 512, ct5, tag5, zpt), 2, 1)
    ms_d = timed(lambda: eng.ed448_key_decrypt_dev(pw, pw_off[: n5 + 1], zpt, ct5, m5_off, tag5, 512, pt5, ok5), 2, 1)
    assert bool(ok5.all().item()) and bool(torch.equal(pt5, m5)), "ECDHIES round trip failed"
    for i in (0, n5 - 1):  # Python big-integer restatement of ecc/encryptable.rs:34-50
        c_ref, t_ref, z_ref = ref_ed448.key_encrypt(ref_ed448.point_from_bytes(pub[i * 112:(i + 1) * 112].cpu().numpy().tobytes()),
                                                    m5[i * 256:(i + 1) * 256].cpu().numpy().tobytes(), 512,
                                                    k_rand[i * 56:(i + 1) * 56].cpu().numpy().tobytes())
        assert ct5[i * 256:(i + 1) * 256].cpu().numpy().tobytes() == c_ref and tag5[i * 56:(i + 1) * 56].cpu().numpy().tobytes() == t_ref
        assert zpt[i * 112:(i + 1) * 112].cpu().numpy().tobytes() == ref_ed448.point_to_bytes(z_ref), "key_encrypt != oracle"
    out["ed448_ecdhies_2^18x256B"] = {
        "key_encrypts_per_s": world * n5 / (ms_e * 1e-3), "key_decrypts_per_s": world * n5 / (ms_d * 1e-3),
        "ms_encrypt": ms_e, "ms_decrypt": ms_d,
        "note": "encrypt = 1 variable-base + 1 fixed-base scalar mult + 3 KMACs, decrypt = 1 variable-base + 4 KMACs"}

    # e2e for the Ed448 half of the metric: host buffers through capy_ed448_fixed_base_batch (H2D 56 B, D2H 112 B per item)
    # at cfg 3's size (2^20 scalars: four chunks of 2^18 on the ctx's three streams)
    n6 = n3
    h_sc = eng.pinned(n6 * 56)
    h_sc[:] = sc[: n6 * 56].cpu().numpy()
    h_pts = eng.pinned(n6 * 112).reshape(n6, 112)
    dt = timed_host(lambda: eng.ed448_fixed_base(h_sc, out=h_pts), 3)
    assert np.array_equal(h_pts[idx3], rows(pts, n3, 112, idx3).reshape(NS, 112)), "cfg 3 e2e != device-resident result"
    out["ed448_fixed_base_e2e_2^20"] = {"scalar_mults_per_s": world * n6 / dt, "ms_per_step": dt * 1e3,
                                        "h2d_bytes_per_step": n6 * 56, "d2h_bytes_per_step": n6 * 112,
                                        "api": "capy_ed448_fixed_base_batch (pinned host buffers from capy_host_alloc)"}
    eng.set_plan_cache(False)
    return out


if __name__ == "__main__":
    main()
