"""pcls_dataset_stats and DatasetStats on the GPU: the kernel against the float64 oracle (oracle/dataset_stats.py) for
float32 / float64 input with 5 and 6 channels at the benchmark shapes and an odd one, bit-identical per-frame rows
whatever the batch, raw scans equal to the .npy files the converter writes from them, and N GPUs equal to one."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import dataset_stats as O
from tests.util import synth_range_images, synth_scan

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NC = 20
SHIFT = np.array([-0.047, 0.365, -0.855, 0.2198, 8.3568])    # KITTI INPUT_MEAN


def _frames(rng, B, H, W, channels, dtype):
  """Synthetic frames with every invalid-pixel kind, labels outside [0, NC) and one all-invalid frame."""
  f = synth_range_images(rng, B, H, W, valid_rate=0.7, channels=channels, num_classes=NC).astype(np.float64)
  f[..., :4] += rng.normal(0, 1e-3, f[..., :4].shape) * (f[..., 4:5] > 0)   # values that are not float32-round
  depth = f[..., 4]
  k = rng.random(depth.shape)
  depth[k < 0.03] = -rng.uniform(0.1, 5, int((k < 0.03).sum()))          # negative range
  depth[(k >= 0.03) & (k < 0.05)] = np.nan                                # NaN range
  f[(k >= 0.05) & (k < 0.07), :4] = np.nan                                # NaN values at range-0 pixels
  f[(k >= 0.05) & (k < 0.07), 4] = 0.0
  if channels == 6:
    lab = f[..., 5]
    u = rng.random(lab.shape)
    lab[u < 0.02] = rng.uniform(-3, 0, int((u < 0.02).sum()))              # (-1, 0) truncates to 0, <= -1 dropped
    lab[(u >= 0.02) & (u < 0.04)] = NC + rng.integers(0, 100, int(((u >= 0.02) & (u < 0.04)).sum()))
    lab[(u >= 0.04) & (u < 0.05)] = np.nan
    lab[(u >= 0.05) & (u < 0.055)] = np.inf
    lab[(u >= 0.055) & (u < 0.1)] += 0.75                                  # fractional: truncated
  if B > 1:
    f[1, ..., 4] = 0.0                                                     # all-invalid frame
  return f.astype(dtype)


def _kernel(frames, shift=SHIFT, labels=True):
  """Runs pcls_dataset_stats once on a CUDA tensor; returns numpy outputs."""
  from pclsegmentation_b200 import _lib
  B, H, W, C = frames.shape
  dev = frames.device
  sums = torch.empty((B, 5, 4), dtype=torch.float64, device=dev)
  valid = torch.empty(B, dtype=torch.int64, device=dev)
  row, col = torch.zeros(H, dtype=torch.int64, device=dev), torch.zeros(W, dtype=torch.int64, device=dev)
  cls, drop = torch.zeros(NC, dtype=torch.int64, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
  lab = labels and C == 6
  sh = np.ascontiguousarray(shift, np.float64)
  _lib.check(_lib.load().pcls_dataset_stats(
      frames.data_ptr(), 1 if frames.dtype == torch.float64 else 0, C, B, H, W,
      sh.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), NC, sums.data_ptr(), valid.data_ptr(), row.data_ptr(),
      col.data_ptr(), cls.data_ptr() if lab else None, drop.data_ptr() if lab else None,
      torch.cuda.current_stream().cuda_stream), "pcls_dataset_stats")
  torch.cuda.synchronize()
  return dict(frame_sums=sums.cpu().numpy(), frame_valid=valid.cpu().numpy(), row_valid=row.cpu().numpy(),
              col_valid=col.cpu().numpy(), class_pixels=cls.cpu().numpy(), dropped=int(drop.item()))


@pytest.mark.parametrize("H,W,B", [(64, 2048, 3), (32, 1024, 4), (32, 240, 5), (7, 33, 9)])
@pytest.mark.parametrize("channels", [5, 6])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_kernel_matches_oracle(H, W, B, channels, dtype):
  from pclsegmentation_b200.dataset_stats import DatasetStats
  rng = np.random.default_rng(H * 1000 + W + channels)
  f = _frames(rng, B, H, W, channels, dtype)
  got = _kernel(torch.from_numpy(f).cuda())
  ref = O.frame_stats(f, SHIFT, NC)
  for k in ("frame_valid", "row_valid", "col_valid"):
    assert np.array_equal(got[k], ref[k]), k
  assert got["frame_valid"][1] == 0
  assert np.array_equal(got["frame_sums"][:, :, 2:], ref["frame_sums"][:, :, 2:])          # min / max exact
  assert (got["frame_sums"][1, :, :2] == 0).all() and (got["frame_sums"][1, :, 2] == np.inf).all()
  assert (got["frame_sums"][1, :, 3] == -np.inf).all()
  n = ref["frame_valid"][:, None]
  np.testing.assert_allclose(got["frame_sums"][:, :, 1], ref["frame_sums"][:, :, 1], rtol=1e-12)
  scale = np.sqrt(n * ref["frame_sums"][:, :, 1]) + 1e-300                                   # |sum(d)| <= this
  assert (np.abs(got["frame_sums"][:, :, 0] - ref["frame_sums"][:, :, 0]) <= 1e-12 * scale).all()
  if channels == 6:
    assert np.array_equal(got["class_pixels"], ref["class_pixels"]) and got["dropped"] == ref["dropped"] > 0
  else:
    assert not got["class_pixels"].any() and got["dropped"] == 0
  # the whole set through DatasetStats: mean / std of every valid pixel
  st = DatasetStats(NC, H, W, shift=SHIFT)
  st.update(f)
  rep = st.finish()
  mean, std = O.dataset_moments(f)
  # rtol 1e-12, and 1e-12 of the channel's spread for means near 0 (y of a symmetric scan: |mean| ~ 1e-4 while both
  # sides carry rounding at the scale of the values)
  assert (np.abs(rep["mean"].reshape(5) - mean) <= 1e-12 * (np.abs(mean) + std)).all(), (rep["mean"], mean)
  np.testing.assert_allclose(rep["std"].reshape(5), std, rtol=1e-12)
  assert rep["valid"] == int(ref["frame_valid"].sum()) and rep["frames"] == B
  assert np.array_equal(rep["min"], ref["frame_sums"][:, :, 2].min(0))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_nan_value_at_a_valid_pixel_enters_the_sums_not_min_max(dtype):
  rng = np.random.default_rng(21)
  f = _frames(rng, 3, 7, 33, 6, dtype)
  vy, vx = np.nonzero(f[0, ..., 4] > 0)
  f[0, vy[0], vx[0], 0] = np.nan                          # x of one valid pixel
  f[2, vy[1], vx[1], 1] = np.nan                          # y of another, in another frame
  got = _kernel(torch.from_numpy(f).cuda())
  ref = O.frame_stats(f, SHIFT, NC)
  assert np.isnan(got["frame_sums"][0, 0, :2]).all() and np.isnan(got["frame_sums"][2, 1, :2]).all()
  assert not np.isnan(got["frame_sums"][:, :, 2:]).any()
  assert np.array_equal(got["frame_sums"][:, :, 2:], ref["frame_sums"][:, :, 2:])          # NaN left out of min / max
  np.testing.assert_allclose(got["frame_sums"][:, :, 1], ref["frame_sums"][:, :, 1], rtol=1e-12)   # NaN == NaN
  assert np.array_equal(got["frame_valid"], ref["frame_valid"])


def test_frame_rows_do_not_depend_on_the_batch():
  rng = np.random.default_rng(11)
  H, W = 64, 2048
  x = _frames(rng, 1, H, W, 6, np.float64)[0]
  rows = []
  for B, pos in ((1, 0), (7, 5), (64, 63)):
    batch = torch.empty((B, H, W, 6), dtype=torch.float64, device="cuda")
    batch.uniform_(1.0, 50.0)
    batch[pos] = torch.from_numpy(x).cuda()
    r = _kernel(batch)
    rows.append(r["frame_sums"][pos].tobytes())
    if B == 7:
      again = _kernel(batch)
      assert again["frame_sums"].tobytes() == r["frame_sums"].tobytes()
      assert np.array_equal(again["row_valid"], r["row_valid"]) and np.array_equal(again["col_valid"], r["col_valid"])
    del batch
  assert rows[0] == rows[1] == rows[2]


def test_finish_does_not_depend_on_the_batch_size():
  from pclsegmentation_b200.dataset_stats import DatasetStats
  rng = np.random.default_rng(12)
  f = _frames(rng, 64, 32, 1024, 6, np.float64)
  reps = []
  for batch in (1, 16, 64):
    st = DatasetStats(NC, 32, 1024, shift=SHIFT)
    for i in range(0, 64, batch):
      st.update(f[i:i + batch])
    reps.append({k: (v.tobytes() if isinstance(v, np.ndarray) else v) for k, v in st.finish().items()})
  assert reps[0] == reps[1] == reps[2]


def test_raw_scans_equal_the_converted_files(tmp_path):
  from pclsegmentation_b200 import dataset_convert, dataset_stats
  rng = np.random.default_rng(13)
  scans_dir = tmp_path / "scans"
  scans_dir.mkdir()
  for i in range(5):
    n = int(rng.integers(20000, 40000))
    synth_scan(rng, n).tofile(str(scans_dir / ("%06d.bin" % i)))
    (rng.integers(0, 26, n).astype(np.uint32) | (rng.integers(0, 9, n).astype(np.uint32) << 16)).tofile(
        str(scans_dir / ("%06d.label" % i)))
  common = ["--labels", str(scans_dir / "*.label"), "--width", "512"]
  dataset_convert.main(["--scans", str(scans_dir / "*.bin"), "--output_dir", str(tmp_path / "npy"), "--batch", "2"]
                       + common)
  from_files = dataset_stats.main(["-d", str(tmp_path / "npy" / "*.npy"), "-b", "3", "--json", str(tmp_path / "a.json")])
  from_scans = dataset_stats.main(["--scans", str(scans_dir / "*.bin"), "-b", "4"] + common)
  assert from_files["frames"] == 5 and from_files["dropped"] > 0 and from_files["class_pixels"].sum() > 0
  for k, v in from_files.items():
    w = from_scans[k]
    assert (v.tobytes() == w.tobytes()) if isinstance(v, np.ndarray) else v == w, k
  assert set(json.load(open(tmp_path / "a.json"))) == set(dataset_stats.KEYS)
  # scans without label files: the converter fills the label channel with 0; -d --no_labels skips it like --scans
  dataset_convert.main(["--scans", str(scans_dir / "*.bin"), "--output_dir", str(tmp_path / "nolab"), "--width", "512"])
  a = dataset_stats.main(["-d", str(tmp_path / "nolab" / "*.npy"), "--no_labels"])
  b = dataset_stats.main(["--scans", str(scans_dir / "*.bin"), "--width", "512"])
  assert a["class_pixels"].sum() == b["class_pixels"].sum() == 0 and a["dropped"] == b["dropped"] == 0
  assert a["mean"].tobytes() == b["mean"].tobytes() == from_files["mean"].tobytes()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_n_gpus_equal_one():
  n = min(torch.cuda.device_count(), 8)
  cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr",
         "127.0.0.1", "--master-port", "29519", os.path.join(ROOT, "tests", "multi_gpu_dataset_stats_worker.py")]
  r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
  rep = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
  assert rep["ok"] and rep["world"] == n
