"""-m gpu: `bench.py --dump-outputs` saves what the last timed step computed as float32 .npy files (at most 64 MB),
and two runs with the same arguments but different step counts save the same arrays (seeded weights and inputs;
weight gradients up to the order of their atomic accumulation)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(cwd, steps, dump_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--image", "2048", "--no-cpu-baseline", "--no-cudnn-baseline", "--dump-outputs", str(dump_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=cwd)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_dump_outputs_are_reproducible(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    assert _bench(tmp_path, 2, a)["steps"] == 2
    assert _bench(tmp_path, 3, b)["steps"] == 3
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    # the weight gradients, the step's result, and per distinct layer (27) its output and, past the first, its input gradient
    assert len(names) == 2 + 27 + 26 and "weight_grads.npy" in names and "step_result.npy" in names
    layers = json.load(open(os.path.join(ROOT, "tests", "golden", "layers_amoebanetd_sp4.json")))["layers"]
    assert np.load(a / "weight_grads.npy").size == sum(l["K"] * l["C"] * l["R"] * l["S"] for l in layers if l["op"] == "conv")
    total = 0
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype == np.float32 and np.isfinite(x).all() and np.abs(x).max() > 0, n
        if n == "weight_grads.npy":
            # the wgrad kernels add fp32 partial sums of pixel blocks atomically, in an order that varies from run to run
            np.testing.assert_allclose(x, y, rtol=2e-2, atol=1e-2 * np.abs(x).max(), err_msg=n)
        else:
            np.testing.assert_array_equal(x, y, err_msg=n)
        total += x.nbytes
    assert total <= 64 << 20
