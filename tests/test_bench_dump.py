"""CPU: bench.py --dump-outputs writes the step's results as float32 / float64 .npy files within 64 MB, sampling
images with a fixed seed when the batch is too large."""
import os

import numpy as np

import bench


def _outputs(batch):
    rng = np.random.default_rng(3)
    return {"loss_result": rng.normal(size=16), "kept": rng.integers(-1, 8732, (batch, 80, 200)).astype(np.int32),
            "count": rng.integers(0, 200, (batch, 80)).astype(np.int32)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_whole_batch_is_written_exactly(tmp_path):
    out = _outputs(8)
    bench.write_outputs(str(tmp_path), out)
    got = _load(str(tmp_path))
    assert sorted(got) == ["count", "kept", "loss_result"]
    assert got["loss_result"].dtype == np.float64 and np.array_equal(got["loss_result"], out["loss_result"])
    for k in ("kept", "count"):
        assert got[k].dtype == np.float32 and np.array_equal(got[k], out[k])


def test_large_batch_is_sampled_under_the_limit(tmp_path):
    out = _outputs(1100)
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), out)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))) <= 64 << 20
    images = a["images"].astype(np.int64)
    assert 0 < images.size < 1100 and np.all(np.diff(images) > 0)
    assert np.array_equal(a["kept"], out["kept"][images]) and np.array_equal(a["count"], out["count"][images])
    assert all(np.array_equal(a[k], b[k]) for k in a)
