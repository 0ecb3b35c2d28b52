"""bench.py on the GPU: `--steps K` times exactly K steps, and `--dump-outputs` writes what the last of them returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_the_last_timed_step(tmp_path):
    cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--steps", "3", "--warmup", "3", "--regions", "2", "--no-cpu-baseline",
           "--no-extra", "--no-parity", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    assert line["steps"] == 3 and line["timed_region_steps"] == [2, 1]
    y, idx = np.load(tmp_path / "waveform.npy"), np.load(tmp_path / "indices.npy")
    assert y.dtype == np.float32 and y.shape == (64, 1, 48000)
    assert idx.dtype == np.float64 and idx.shape == (8, 64, 160)
    # bench's inputs are four batches drawn from seed 1337 and timed step i reads batch i % 4, so the last of 3 steps read batch 2;
    # a 1 s step's output depends on its own input and the tail of the step before, so a fresh codec fed batches 1, 2 must agree
    import bench
    gen = torch.Generator().manual_seed(1337)
    xs = [0.1 * torch.randn(64, 1, 48000, generator=gen) for _ in range(3)]
    dev = torch.device("cuda:0")
    tx, rx, dec = bench.build_codec("symad", dev)
    bench.codec_step(tx, rx, dec, xs[1].to(dev))
    ry, ridx = bench.codec_step(tx, rx, dec, xs[2].to(dev))
    np.testing.assert_array_equal(idx, ridx.cpu().numpy())
    np.testing.assert_array_equal(y, ry.cpu().numpy())
