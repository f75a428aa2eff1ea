"""bench.py --dump-outputs: the outputs of the last timed step of the default workload land in the given directory as
float32 .npy files, large outputs as a fixed sample, within 64 MB."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_last_step_outputs(tmp_path):
    out = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "linear", "--profile",
           "--steps", "2", "--warmup", "1", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    arrs = {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}
    assert sorted(arrs) == ["bias_grad", "input_grad", "output", "weight_grad"]
    assert sum(a.nbytes for a in arrs.values()) <= 64 << 20
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrs.values())
    assert arrs["output"].shape == arrs["input_grad"].shape == arrs["weight_grad"].shape == (1 << 20,)
    # backward(1 / (n * fout)) seeds every element of dY with the same value, so db = n / (n * fout) = 1 / fout
    assert arrs["bias_grad"].shape == (4096,) and np.allclose(arrs["bias_grad"], 1 / 4096, rtol=1e-6, atol=0)
