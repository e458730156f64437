"""bench.py --dump-outputs: what the timed path computed in its last step, as float32 .npy files."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT, rel_err


def test_dump_keeps_small_arrays_and_a_fixed_sample_of_large_ones(tmp_path):
    small = torch.arange(12, dtype=torch.float64).reshape(3, 4)
    large = torch.arange(bench.DUMP_SAMPLE + 1000, dtype=torch.float32).reshape(-1, 8)  # element i holds i
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"small": small, "large": large, "half": small.to(torch.bfloat16)})
    for name in ("small", "half"):
        got = np.load(tmp_path / "a" / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == (3, 4) and np.array_equal(got, small.numpy())
    a, b = np.load(tmp_path / "a" / "large.npy"), np.load(tmp_path / "b" / "large.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_SAMPLE,) and np.array_equal(a, b)
    assert (np.diff(a) > 0).all() and a[0] >= 0 and a[-1] < large.numel()  # distinct elements, in memory order
    # one sample element per output array, four arrays: within 64 MB in all
    assert len(bench.OUTPUT_NAMES) * bench.DUMP_SAMPLE * 4 <= 64 << 20


@pytest.mark.gpu
def test_dump_is_the_op_on_the_seeded_inputs(tmp_path):
    """The dumped arrays are the op's output and gradients for the seeded config-2 batch, and --steps/--warmup are the
    numbers of timed and untimed steps the line reports."""
    from weed_instance_segmentation_b200 import build
    build.build()
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--no-extras", "--no-train",
           "--no-cpu-baseline", "--no-gpu-reference", "--dump-outputs", str(tmp_path / "bench")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["warmup"] == 1
    prob = bench.Problem("init", "bf16", torch.device("cuda", 0), seed=0)
    prob.step()
    torch.cuda.synchronize()
    bench.dump_outputs(str(tmp_path / "fresh"), dict(zip(bench.OUTPUT_NAMES, (prob.out, prob.gv, prob.gl, prob.ga))))
    total = 0
    for name in bench.OUTPUT_NAMES:
        got, want = np.load(tmp_path / "bench" / f"{name}.npy"), np.load(tmp_path / "fresh" / f"{name}.npy")
        total += os.path.getsize(tmp_path / "bench" / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == want.shape, name
        assert np.abs(want).max() > 0, name
        if name == "output":
            assert np.array_equal(got, want)
        else:  # bf16 gradients accumulated in float32: the order of the additions may differ between two calls
            assert rel_err(got, want) <= 1e-2, name
    assert total <= 64 << 20
