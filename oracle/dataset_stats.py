"""Dataset statistics of range images in numpy float64: the contract of ``pcls_dataset_stats`` (include/pclseg.h) and of
``DatasetStats.finish``, stated pixel by pixel.

A pixel is valid when its range channel (4) is > 0 (NaN is not).  Over the valid pixels of each frame: sum(x - s),
sum((x - s)^2), min(x), max(x) per channel, with NaN values left out of min / max; valid pixels per row and per
column; the label channel (6-channel frames) truncated toward zero and counted per class, or in ``dropped`` when it is
not finite or not in [0, num_classes)."""
import numpy as np


def frame_stats(frames, shift=None, num_classes=None):
  """frames [B,H,W,5|6] -> dict(frame_sums [B,5,4], frame_valid [B], row_valid [H], col_valid [W], class_pixels [NC],
  dropped); the class outputs only for 6-channel frames with num_classes given."""
  x = np.asarray(frames, dtype=np.float64)
  B, H, W, C = x.shape
  s = np.zeros(5) if shift is None else np.asarray(shift, np.float64).reshape(5)
  with np.errstate(invalid="ignore"):
    valid = x[..., 4] > 0
  sums = np.empty((B, 5, 4))
  for b in range(B):
    v = x[b][valid[b]][:, :5]
    d = v - s
    sums[b, :, 0] = d.sum(0)
    sums[b, :, 1] = (d * d).sum(0)
    sums[b, :, 2] = np.where(np.isnan(v), np.inf, v).min(0, initial=np.inf)
    sums[b, :, 3] = np.where(np.isnan(v), -np.inf, v).max(0, initial=-np.inf)
  out = dict(frame_sums=sums, frame_valid=valid.reshape(B, -1).sum(1).astype(np.int64),
             row_valid=valid.sum((0, 2)).astype(np.int64), col_valid=valid.sum((0, 1)).astype(np.int64))
  if C == 6 and num_classes is not None:
    lab = x[..., 5][valid]
    with np.errstate(invalid="ignore"):
      t = np.trunc(lab)
      ok = np.isfinite(lab) & (t >= 0) & (t < num_classes)
    out["class_pixels"] = np.bincount(t[ok].astype(np.int64), minlength=num_classes).astype(np.int64)
    out["dropped"] = int((~ok).sum())
  return out


def dataset_moments(frames):
  """Per-channel mean and population std over every valid pixel of every frame, straight from the values."""
  x = np.asarray(frames, dtype=np.float64)
  with np.errstate(invalid="ignore"):
    v = x[x[..., 4] > 0][:, :5]
  return v.mean(0), v.std(0)
