"""bench.py --dump-outputs: what it writes is what the timed path computed, so that two builds can be compared output
for output."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
import oracle_lib as o

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_pairings_of_the_benchmark_inputs(ctx, tmp_path):
    """a 2^12 batch (above the latency path's limit: the lane-pair kernel of the headline; every row dumped): the float64
    words decode to the oracle's pairings of bench.make_inputs' points"""
    n = 1 << 12
    r = subprocess.run([sys.executable, bench.__file__, "--batch-log2", "12", "--steps", "2", "--warmup", "1", "--no-secondary",
                        "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["pairing.npy", "pairing_rows.npy"]
    words, rows = np.load(tmp_path / "pairing.npy"), np.load(tmp_path / "pairing_rows.npy")
    assert words.dtype == rows.dtype == np.float64 and words.shape == (n, 144)
    assert np.array_equal(rows, np.arange(n))
    assert (words == np.floor(words)).all() and words.min() >= 0 and words.max() < 2**32
    got = words.astype(np.uint32).view(np.uint64)
    from pairing_b200.device import DeviceEngine
    pa, qa, _, _ = bench.make_inputs(DeviceEngine(ctx=ctx, device=0), n, bench.SEED, torch, np)
    idx = np.arange(0, n, 32)
    pa, qa = pa.cpu().numpy().view(np.uint64)[idx], qa.cpu().numpy().view(np.uint64)[idx]
    assert np.array_equal(got[idx], o.pairing(pa, qa, o.default_threads()))
