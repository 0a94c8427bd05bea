"""bench.py --dump-outputs: file names, dtypes, the size limit and the seeded sample.  CPU only."""
import os

import numpy as np
import torch

import bench


def test_host_outputs_names_and_dtypes():
    """Each gradient lands under the name of the leaf it belongs to (distinct fill values tell them apart)."""
    grads = [torch.full((4, 3, 5, 2, 1), 1.0)] + [torch.full((4, 5, 8), float(i)) for i in range(2, 6)]
    out = bench.host_outputs(torch.tensor(0.5), grads)
    assert bench.GRAD_OUTPUTS == ("fake", "h_fake", "m_real", "h_real", "m_fake")
    assert list(out) == ["loss", "grad_fake", "grad_h_fake", "grad_m_real", "grad_h_real", "grad_m_fake"]
    assert out["loss"].shape == () and float(out["loss"]) == 0.5
    assert all(a.dtype == np.float32 for a in out.values())
    for name, g in zip(bench.GRAD_OUTPUTS, grads):
        assert np.array_equal(out["grad_" + name], g.numpy()), name


def test_dump_whole_arrays_under_the_limit(tmp_path):
    arrays = {"loss": np.float32(1.0).reshape(()), "grad_fake": np.arange(3 * bench.DUMP_SAMPLE, dtype=np.float32)}
    bench.dump_outputs(str(tmp_path / "d"), arrays)
    assert sorted(os.listdir(tmp_path / "d")) == ["grad_fake.npy", "loss.npy"]
    assert np.array_equal(np.load(tmp_path / "d" / "grad_fake.npy"), arrays["grad_fake"])


def test_dump_samples_the_same_elements_above_the_limit(tmp_path):
    n = bench.DUMP_LIMIT_BYTES // 4 + 1
    arrays = {"loss": np.float32(1.0).reshape(()), "grad_fake": np.arange(n, dtype=np.float32),
              "grad_h_fake": np.ones((64, 10, 8), dtype=np.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= bench.DUMP_LIMIT_BYTES
    a, b = np.load(tmp_path / "a" / "grad_fake.npy"), np.load(tmp_path / "b" / "grad_fake.npy")
    assert a.shape == (bench.DUMP_SAMPLE,) and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0)                        # distinct elements, in index order
    assert np.array_equal(np.load(tmp_path / "a" / "grad_h_fake.npy"), arrays["grad_h_fake"])
