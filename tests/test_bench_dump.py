"""CPU: bench.py --dump-outputs writes float32 .npy files that stay under 64 MB for the default workload
and are identical from run to run for identical results (the sample of a large output is fixed)."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_budget_and_fixed_sample(tmp_path):
    g = torch.Generator().manual_seed(0)
    outs = dict(mask_scores=torch.rand(64, 512, 512, 2, generator=g),          # c2: 64 tiles of 512^2
                image_embeddings=torch.rand(64, 256, 32, 32, generator=g),
                topo_scores=torch.rand(64, 256, 16, 1, generator=g), absent=None)
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), outs)
    bench.dump_outputs(str(b), outs)
    names = sorted(os.listdir(a))
    assert names == ["image_embeddings.npy", "mask_scores.npy", "topo_scores.npy"]
    assert sum(os.path.getsize(a / n) for n in names) <= 64 << 20
    for n in names:
        x = np.load(a / n)
        assert x.dtype == np.float32 and np.array_equal(x, np.load(b / n))
    assert np.array_equal(np.load(a / "topo_scores.npy"), outs["topo_scores"].numpy())     # small: stored whole
    sample = np.load(a / "mask_scores.npy")
    assert sample.size == bench.DUMP_MAX_VALUES and np.isin(sample[:100], outs["mask_scores"].numpy()).all()
