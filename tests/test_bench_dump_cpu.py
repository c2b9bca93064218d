"""bench.py --dump-outputs: float64 / float32 .npy files, 64 MB in all, the same seeded sample of an oversized output on
every run."""
import numpy as np
import torch

import bench


def test_dump_outputs_dtypes_cap_and_fixed_sample(tmp_path):
    clouds = torch.randn(4, 2048, 3, dtype=torch.float64)
    weights = torch.randn(10_000_000).bfloat16()  # 40 MB as float32: over its share of the cap
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"samples": clouds, "loss": torch.tensor(0.5), "parameters": weights})
    files = sorted((tmp_path / "a").iterdir())
    assert [f.name for f in files] == ["loss.npy", "parameters.npy", "samples.npy"]
    assert sum(f.stat().st_size for f in files) <= bench.DUMP_BYTES
    s = np.load(tmp_path / "a" / "samples.npy")
    assert s.dtype == np.float64 and np.array_equal(s, clouds.numpy())
    loss = np.load(tmp_path / "a" / "loss.npy")
    assert loss.dtype == np.float32 and loss.tolist() == [0.5]
    p = np.load(tmp_path / "a" / "parameters.npy")
    assert p.dtype == np.float32 and 0 < p.size < weights.numel()
    assert np.isin(p, weights.float().numpy()).all()
    assert np.array_equal(p, np.load(tmp_path / "b" / "parameters.npy"))
