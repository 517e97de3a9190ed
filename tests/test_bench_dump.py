"""bench.py --dump-outputs: the files two builds are compared by (CPU tensors stand in for the device outputs)."""
import numpy as np
import torch

import bench


def _outputs(B, H, W, nc, seed):
  probs = torch.rand((B, H, W, nc), generator=torch.Generator().manual_seed(seed))
  return {"predictions": probs.argmax(-1).to(torch.int32), "probabilities": probs}


def _load(d):
  return {k: np.load(str(d / (k + ".npy"))) for k in ("pixel_index", "predictions", "probabilities")}


def test_every_pixel_when_it_fits(tmp_path):
  res = _outputs(2, 4, 8, 5, 0)
  bench.dump_outputs(str(tmp_path), res)
  got = _load(tmp_path)
  assert got["pixel_index"].dtype == np.float64 and np.array_equal(got["pixel_index"], np.arange(64))
  assert got["predictions"].dtype == np.float32
  assert np.array_equal(got["predictions"], res["predictions"].reshape(-1).numpy())
  assert got["probabilities"].dtype == np.float32
  assert np.array_equal(got["probabilities"], res["probabilities"].reshape(64, 5).numpy())


def test_fixed_sample_within_the_byte_cap(tmp_path, monkeypatch):
  monkeypatch.setattr(bench, "DUMP_BYTES", 40000)
  res = _outputs(4, 16, 64, 20, 1)                  # 4096 pixels x 92 bytes: does not fit
  for d in ("a", "b"):
    bench.dump_outputs(str(tmp_path / d), _outputs(4, 16, 64, 20, 1))
  a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
  assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 40000
  for k in a:
    assert np.array_equal(a[k], b[k]), k
  idx = a["pixel_index"].astype(np.int64)
  assert 0 < len(idx) < 4096 and (np.diff(idx) > 0).all()
  assert np.array_equal(a["predictions"], res["predictions"].reshape(-1).numpy()[idx])
  assert np.array_equal(a["probabilities"], res["probabilities"].reshape(-1, 20).numpy()[idx])
