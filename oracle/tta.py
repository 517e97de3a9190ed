"""Test-time augmentation: a numpy restatement of the contract of pcls_tta_views / pcls_tta_merge (include/pclseg.h).

A view (flip, shift) maps source column w to (flip ? W-1-w : w) + shift mod W, negates y under the mirror and rotates
(x, y) about z by alpha = -2 pi shift / W (not at all for shift 0).  Every float64 operation below is one IEEE
operation with its own rounding, as the device spells it; the 16-bit rounding of the network input goes through numpy
(fp16) or torch (bf16), both round to nearest even."""
import math

import numpy as np
import torch


def rotation(shift, W):
  """(cos, sin) of alpha = -2 pi shift / W in float64; exactly 0 / +-1 when shift is a multiple of W / 4."""
  if (4 * shift) % W == 0:
    return ((1.0, 0.0), (0.0, -1.0), (-1.0, 0.0), (0.0, 1.0))[(4 * shift // W) % 4]
  a = -2.0 * math.pi * shift / W
  return math.cos(a), math.sin(a)


def columns(flip, shift, W):
  """[W] int: the view column of every source column."""
  w = np.arange(W)
  return ((W - 1 - w if flip else w) + shift) % W


def inverse_columns(flip, shift, W):
  """[W] int: the source column of every view column."""
  c = (np.arange(W) - shift) % W
  return W - 1 - c if flip else c


def view_points(x, y, flip, shift, W):
  """float32 x, y -> float64 x', y' of the view (the mirror, then the rotation)."""
  xd = np.asarray(x, np.float32).astype(np.float64)
  yd = (-np.asarray(y, np.float32) if flip else np.asarray(y, np.float32)).astype(np.float64)
  if shift == 0:
    return xd, yd
  c, s = rotation(shift, W)
  return c * xd - s * yd, s * xd + c * yd


def to16(f32, precision):
  """float32 -> uint16 bit patterns of fp16 / bf16 (round to nearest even)."""
  f32 = np.ascontiguousarray(f32, np.float32)
  if precision == "f16":
    return f32.astype(np.float16).view(np.uint16)
  return torch.from_numpy(f32).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def views_input(raw, mean, std, views, precision):
  """raw [B,H,W,5|6] float32, views [(flip, shift), ...] -> (input [T*B,H,W,8] uint16, mask [T*B,H,W] uint8), frame
  t*B + b = view t of frame b."""
  raw = np.asarray(raw, np.float32)
  B, H, W, _ = raw.shape
  mean = np.asarray(mean, np.float64).reshape(-1)[:5]
  std = np.asarray(std, np.float64).reshape(-1)[:5]
  m = raw[..., 4] > 0
  out = np.zeros((len(views) * B, H, W, 8), np.uint16)
  mask = np.zeros((len(views) * B, H, W), np.uint8)
  for t, (flip, shift) in enumerate(views):
    xd, yd = view_points(raw[..., 0], raw[..., 1], flip, shift, W)
    vals = [xd, yd] + [raw[..., c].astype(np.float64) for c in (2, 3, 4)]
    f = np.zeros((B, H, W, 8), np.float32)
    for c in range(5):
      f[..., c] = np.where(m, ((vals[c] - mean[c]) / std[c]).astype(np.float32), np.float32(0))
    f[..., 5] = m.astype(np.float32)
    col = columns(flip, shift, W)
    frame = np.zeros_like(f)
    frame[:, :, col] = f
    out[t * B:(t + 1) * B] = to16(frame, precision)
    mv = np.zeros((B, H, W), np.uint8)
    mv[:, :, col] = m
    mask[t * B:(t + 1) * B] = mv
  return out, mask


def argmax_first(p):
  """[..., NC] float32 -> argmax with the head's rule: `v > best` from best = -1, so the first index wins ties (and a
  NaN never wins)."""
  best = np.zeros(p.shape[:-1], np.int32)
  bp = np.full(p.shape[:-1], np.float32(-1.0), np.float32)
  for c in range(p.shape[-1]):
    up = p[..., c] > bp
    best = np.where(up, c, best)
    bp = np.where(up, p[..., c], bp)
  return best


def merge(probs, mask, views, none_index):
  """probs [T*B,H,W,NC] float32 of the views, mask [T*B,H,W] -> (mean probabilities [B,H,W,NC] float32, predictions
  [B,H,W] int32) on the source pixels: the views summed in view order in float32, divided by T in float32."""
  probs = np.asarray(probs, np.float32)
  T = len(views)
  B = probs.shape[0] // T
  W = probs.shape[2]
  acc = None
  valid = None
  for t, (flip, shift) in enumerate(views):
    col = columns(flip, shift, W)
    p = probs[t * B:(t + 1) * B][:, :, col]
    acc = p.copy() if acc is None else (acc + p).astype(np.float32)
    if t == 0:
      valid = np.asarray(mask)[0:B][:, :, col] != 0
  mean = (acc / np.float32(T)).astype(np.float32)
  pred = np.where(valid, argmax_first(mean), np.int32(none_index)).astype(np.int32)
  return mean, pred
