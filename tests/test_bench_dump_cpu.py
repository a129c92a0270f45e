"""CPU: bench.py --dump-outputs writes the last step's outputs as float32 / float64 .npy files, a fixed seeded sample of
the rays of a large batch, within the 64 MB bound."""
import os

import numpy as np
import torch

import bench


def _outputs(n, s=128):
    g = torch.Generator().manual_seed(n)
    out = {k: torch.rand(n, c, generator=g) for k, c in (("mid_rgb_fine", 3), ("depth_fine", 1))}
    out["weights_fine"] = torch.rand(n, s, 1, generator=g)
    out["mask"] = torch.rand(n, generator=g) > 0.5
    return out


def test_small_batch_is_dumped_whole(tmp_path):
    out = _outputs(64)
    field = torch.nn.Linear(4, 2)
    arrays = bench.step_outputs_to_host(out, torch.tensor(1.5), field)
    bench.dump_step_outputs(arrays, str(tmp_path))
    names = sorted(os.listdir(tmp_path))
    assert names == sorted(["rays.npy", "mid_rgb_fine.npy", "depth_fine.npy", "weights_fine.npy", "mask.npy", "loss.npy",
                            "param.weight.npy", "param.bias.npy"])
    for name in names:
        assert np.load(tmp_path / name).dtype in (np.float32, np.float64), name
    np.testing.assert_array_equal(np.load(tmp_path / "mid_rgb_fine.npy"), out["mid_rgb_fine"].numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "mask.npy"), out["mask"].float().numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "param.weight.npy"), field.weight.detach().numpy())
    assert float(np.load(tmp_path / "loss.npy")) == 1.5


def test_large_batch_is_a_fixed_sample_within_the_bound():
    n = 640000
    out = _outputs(n)
    a, b = bench.step_outputs_to_host(out), bench.step_outputs_to_host(out)
    rays = a["rays"].astype(np.int64)
    assert len(rays) == bench.DUMP_RAYS and np.all(np.diff(rays) > 0) and rays[-1] < n
    np.testing.assert_array_equal(a["rays"], b["rays"])
    np.testing.assert_array_equal(a["mid_rgb_fine"], out["mid_rgb_fine"][rays].numpy())
    np.testing.assert_array_equal(a["weights_fine"], out["weights_fine"][rays[:bench.DUMP_SAMPLE_RAYS]].numpy())
    assert sum(x.nbytes for x in a.values()) <= bench.DUMP_MAX_BYTES
