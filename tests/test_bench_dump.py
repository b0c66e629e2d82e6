"""CPU: bench.py --dump-outputs writes float32 / float64 .npy files within its byte budget, small outputs whole and larger
ones as the same seeded sample on every call."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_budget_dtypes_and_repeatable_sample(tmp_path):
    g = torch.Generator().manual_seed(0)
    y_hat = torch.randn(4, 8, 16, 16, generator=g)
    outs = {"y_hat": y_hat, "means": 2 * y_hat, "log2_lik_sum": torch.tensor([3.5]),
            "symbols": torch.arange(-50, 50, dtype=torch.int32).repeat(40), "likelihoods": {"z": torch.rand(2, 3, 4, generator=g)}}
    budget = 16 << 10
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs, budget=budget)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["likelihoods.z.npy", "log2_lik_sum.npy", "means.npy", "symbols.npy", "y_hat.npy"]
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert sum(v.nbytes for v in a.values()) <= budget
    assert a["y_hat.npy"].dtype == np.float32 and a["symbols.npy"].dtype == np.float64
    np.testing.assert_array_equal(a["likelihoods.z.npy"], outs["likelihoods"]["z"].numpy())
    np.testing.assert_array_equal(a["log2_lik_sum.npy"], [3.5])
    for name in ("y_hat", "symbols"):
        full, sample = outs[name].numpy().ravel(), a[name + ".npy"]
        assert sample.ndim == 1 and 0 < sample.size < full.size
        idx = np.sort(np.random.default_rng(0).choice(full.size, sample.size, replace=False))
        np.testing.assert_array_equal(sample, full[idx])
    np.testing.assert_array_equal(a["means.npy"], 2 * a["y_hat.npy"])        # same-size outputs: the same elements
    for f in files:
        np.testing.assert_array_equal(a[f], np.load(tmp_path / "b" / f))
