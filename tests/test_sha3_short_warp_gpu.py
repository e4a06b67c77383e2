"""The single-block SHA3 kernel (sha3_short_kernel) hashes the 32 messages of a warp together, so its results depend on
how a batch falls into warps.  Batch sizes around warp boundaries (a lone message, a partial first or last warp, an
exact multiple of 32) for every message length the kernel is compiled for, checked against hashlib.  Digests past the
batch must stay unwritten, and rows past the batch must not leak into the digests."""
import hashlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIZES = (1, 31, 32, 33, 127, 129)
CASES = [(256, m) for m in (2, 4, 6, 8, 10, 12, 14, 16)] + [(512, m) for m in (2, 4, 6, 8)]


@pytest.mark.parametrize("d,msg_lanes", CASES)
@pytest.mark.parametrize("pad_stride", (0, 48))
def test_short_kernel_warp_edges(engine, d, msg_lanes, pad_stride):
    import torch

    msg_len = 8 * msg_lanes
    stride = msg_len + pad_stride
    digest = d // 8
    rng = np.random.default_rng(1000 * d + msg_lanes + pad_stride)
    hashf = hashlib.sha3_256 if d == 256 else hashlib.sha3_512
    for n in SIZES:
        rows = n + 40  # rows past n hold data the kernel must not hash
        data = rng.integers(0, 256, size=rows * stride, dtype=np.uint8)
        data[:msg_len] = 0xFF  # all-ones and all-zero messages in the first warp
        data[stride:stride + msg_len] = 0
        guard = 3 * 64
        out = torch.full((n * digest + guard,), 0xA5, dtype=torch.uint8, device="cuda")
        engine.sha3_fixed_dev(torch.from_numpy(data).cuda(), msg_len, stride, n, d, out)
        got = out.cpu().numpy()
        want = b"".join(hashf(data[k * stride:k * stride + msg_len].tobytes()).digest() for k in range(n))
        assert got[:n * digest].tobytes() == want, (n, d, msg_len, stride)
        assert (got[n * digest:] == 0xA5).all(), (n, d, msg_len, stride)
