"""`bench.py --dump-outputs` end to end on the GPU (the CUDA-graph training step and the render workload): the dump holds
the last timed step's outputs, and two runs with the same arguments write the same arrays."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *extra):
    cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--rays", "2048",
           "--no-cpu-baseline", "--no-cuda-baseline", "--dump-outputs", str(out_dir), *extra]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.parametrize("workload", ["train", "render"])
def test_dump_is_the_same_from_run_to_run(tmp_path, workload):
    a = _bench(tmp_path / "a", "--workload", workload)
    b = _bench(tmp_path / "b", "--workload", workload)
    assert "mid_rgb_fine" in a and a["mid_rgb_fine"].shape == (2048, 3)
    if workload == "train":
        assert a["loss"].shape == () and np.isfinite(a["loss"]) and "param.mlp_base.layers.0.weight" in a
    assert sorted(a) == sorted(b)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
