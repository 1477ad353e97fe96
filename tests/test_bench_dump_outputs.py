"""CPU: bench.py --dump-outputs writes float32 .npy files, whole under the size limit and as a fixed sample above it."""
import numpy as np
import torch

import bench


def _outputs():
    return {"pred4": torch.arange(48, dtype=torch.float64).view(2, 1, 4, 6), "prob_volume2": torch.randn(2, 3, 2, 4)}


def test_small_outputs_are_written_whole_in_float32(tmp_path):
    out = _outputs()
    bench.dump_outputs(str(tmp_path), out)
    for name, t in out.items():
        a = np.load(tmp_path / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == tuple(t.shape)
        assert np.array_equal(a, t.float().numpy())


def test_large_outputs_become_the_same_sample_on_every_run(tmp_path):
    out = _outputs()
    limit = 96                                   # bytes; the two arrays hold 384 in float32
    bench.dump_outputs(str(tmp_path / "a"), out, limit)
    bench.dump_outputs(str(tmp_path / "b"), out, limit)
    written = 0
    for name, t in out.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
        assert a.size == t.numel() // 4 and np.isin(a, t.float().numpy()).all()
        written += a.nbytes
    assert written <= limit
