"""CPU: what bench.py writes -- the --dump-outputs sample, and nothing inside the tree (the tree the benchmark runs from
may be read-only)."""
import os

import numpy as np
import torch

import bench
from oracle import cpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_a_seeded_float32_sample(tmp_path):
    digests = torch.randint(0, 256, (bench.N_MSGS * bench.DIGEST,), dtype=torch.uint8, generator=torch.Generator().manual_seed(5))
    bench.dump_outputs(str(tmp_path), digests)
    files = sorted(tmp_path.iterdir())
    assert [f.name for f in files] == ["sha3_256_digests.npy"] and sum(f.stat().st_size for f in files) <= 64e6
    got = np.load(files[0])
    rows = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(bench.N_MSGS, bench.DUMP_ROWS, replace=False))
    assert got.dtype == np.float32 and got.shape == (bench.DUMP_ROWS, bench.DIGEST)
    assert np.array_equal(got, digests.view(bench.N_MSGS, bench.DIGEST).numpy()[rows].astype(np.float32))


def test_native_oracle_is_built_outside_the_tree():
    out = os.path.abspath(cpu.build(native=True))
    assert os.path.exists(out) and not out.startswith(ROOT + os.sep)
