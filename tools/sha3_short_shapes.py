# development aid: every shape of the single-block SHA3 kernel (sha3_short_kernel<17, m> for 16..128-byte messages,
# <9, m> for 16..64-byte messages) over 2^20 messages through capy_sha3_batch_fixed_dev.  One JSON line per shape:
# median ms per launch over 5 windows of 100 launches (CUDA events), GB/s of message bytes, and a SHA-256 of the
# digests so that two builds (CAPY_GPU_LIB) can be compared shape by shape.
import os as _os, sys as _sys
_sys.path.insert(0, _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), '..'))
import hashlib
import json
import statistics

import torch

from capycrypt_b200 import Engine

eng = Engine()
n = 1 << 20
g = torch.Generator(device="cuda")
g.manual_seed(3)
data = torch.randint(0, 256, (n * 128,), dtype=torch.uint8, device="cuda", generator=g)
out = torch.zeros(n * 64, dtype=torch.uint8, device="cuda")
for d, ms in ((256, (2, 4, 6, 8, 10, 12, 14, 16)), (512, (2, 4, 6, 8))):
    for m in ms:
        msg_len = 8 * m
        launch = lambda: eng.sha3_fixed_dev(data, msg_len, msg_len, n, d, out)
        for _ in range(10):
            launch()
        windows = []
        for _ in range(5):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(100):
                launch()
            e1.record()
            torch.cuda.synchronize()
            windows.append(e0.elapsed_time(e1) / 100)
        ms_launch = statistics.median(windows)
        digest = hashlib.sha256(out[:n * d // 8].cpu().numpy().tobytes()).hexdigest()[:16]
        print(json.dumps({"d": d, "msg_len": msg_len, "ms": round(ms_launch, 4), "spread_ms": round(max(windows) - min(windows), 4),
                          "GBps": round(n * msg_len / ms_launch / 1e6, 1), "digests_sha256": digest}), flush=True)
