"""CPU: bench.dump_outputs writes the step's loss and a seeded sample of the flat fp32 weights as float32 .npy, at the
same positions on every call, whole when the buffer is small and within 64 MB at OF-3B size."""
import os
import types

import numpy as np
import torch

import bench


def _bucket(total):
    return types.SimpleNamespace(total=total, device=torch.device("cpu"),
                                 params=torch.arange(total, dtype=torch.float32))


def _dump(path, bucket, **kw):
    bench.dump_outputs(str(path), torch.tensor(2.5, dtype=torch.bfloat16), bucket, **kw)
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_small_buffer_is_written_whole(tmp_path):
    got = _dump(tmp_path, _bucket(1000))
    assert sorted(got) == ["loss", "params"]
    assert got["loss"].dtype == np.float32 and got["loss"].shape == () and got["loss"] == 2.5
    assert got["params"].dtype == np.float32 and np.array_equal(got["params"], np.arange(1000, dtype=np.float32))


def test_large_buffer_is_sampled_at_fixed_distinct_positions(tmp_path):
    bucket = _bucket(1 << 16)
    a = _dump(tmp_path / "a", bucket, sample=4096)["params"]
    b = _dump(tmp_path / "b", bucket, sample=4096)["params"]
    assert a.shape == (4096,) and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0)           # params[i] == i: sorted, distinct positions


def test_of3b_sample_fits_64_mb():
    assert bench.DUMP_SAMPLE * 4 + 4 <= 64 << 20
