"""Test-time augmentation (TTA) on the GPU: mirrored and yaw-rotated views of each raw range image go through one
forward over T x B frames (pcls_tta_views writes them straight into the net's input), and the views' class
probabilities are averaged back onto the source pixels (pcls_tta_merge).  The view and merge rules are in
include/pclseg.h and oracle/tta.py.

Every config trains with RANDOM_FLIPPING and SHIFT_LEFT_RIGHT (configs/_tables.py), so the mirror and horizontal rolls
are views the networks have seen.  TTA needs the RAW input: the normalised 6-channel contract ``model([lidar, mask])``
cannot be un-normalised exactly to negate y, so it is not offered there."""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from .device import ptr, stream_handle

MAX_VIEWS = 8   # include/pclseg.h PCLS_TTA_MAX_VIEWS


def view_rotation(shift, W):
  """(cos, sin) of alpha = -2 pi shift / W in float64; exactly 0 / +-1 when shift is a multiple of W / 4."""
  if (4 * shift) % W == 0:
    return ((1.0, 0.0), (0.0, -1.0), (-1.0, 0.0), (0.0, 1.0))[(4 * shift // W) % 4]
  a = -2.0 * math.pi * shift / W
  return math.cos(a), math.sin(a)


class TTA:
  """The views of test-time augmentation: ``[(f, s) for f in (0, 1 if flip) for s in shifts]``, unflipped first,
  shifts in the given order.  A shift rolls the image by that many columns (the sensor turned by shift / W of a full
  turn; W / 2 is the half turn); ``flip`` adds the mirror image of each.  At most 8 views, no view twice, every shift
  in [0, W)."""

  def __init__(self, flip=True, shifts=(0,)):
    self.flip = bool(flip)
    self.shifts = tuple(int(s) for s in shifts)
    self.view_list = [(f, s) for f in ((0, 1) if self.flip else (0,)) for s in self.shifts]
    if not self.view_list:
      raise ValueError("TTA needs at least one shift")
    if len(self.view_list) > MAX_VIEWS:
      raise ValueError("%d views, at most %d are supported" % (len(self.view_list), MAX_VIEWS))
    if len(set(self.view_list)) != len(self.view_list):
      raise ValueError("a view appears twice in %s" % (self.view_list,))
    if any(s < 0 for s in self.shifts):
      raise ValueError("shifts must be >= 0, got %s" % (self.shifts,))

  def __len__(self):
    return len(self.view_list)

  def __repr__(self):
    return "TTA(flip=%s, shifts=%s)" % (self.flip, self.shifts)

  def views(self, W):
    """(flip int32, shift int32, cos float64, sin float64) arrays of the views for images W columns wide."""
    bad = [s for s in self.shifts if not 0 <= s < W]
    if bad:
      raise ValueError("shifts %s are not in [0, %d)" % (bad, W))
    flip = np.array([f for f, _ in self.view_list], np.int32)
    shift = np.array([s for _, s in self.view_list], np.int32)
    cs = np.array([view_rotation(s, W) for _, s in self.view_list], np.float64).reshape(-1, 2)
    return flip, shift, cs[:, 0].copy(), cs[:, 1].copy()


def parse_shifts(text):
  """``--tta_shifts 0,1024`` -> (0, 1024)."""
  return tuple(int(s) for s in str(text).split(",") if s.strip())


def from_args(flip, shifts):
  """The CLIs' ``--tta`` / ``--tta_shifts``: None (no TTA, the plain path) when neither is given."""
  if not flip and shifts is None:
    return None
  return TTA(flip=flip, shifts=parse_shifts(shifts) if shifts is not None else (0,))


def _c_array(ctype, values):
  return (ctype * len(values))(*[v.item() if hasattr(v, "item") else v for v in values])


def forward_tta(model, raw, tta, want_probabilities=False, out=None):
  """raw [B,H,W,5|6] float32 CUDA range images (x, y, z, remission, range[, label]; mean / std from ``model.mc``) ->
  dict(predictions [B,H,W] int32, probabilities [B,H,W,NC] float32 when asked) merged over the views of ``tta``.
  The net runs one forward over T x B frames: staged in its own input buffers when they hold T x B frames, otherwise
  (a ``micro_batch`` option) through a 16-bit [T x B,H,W,8] tensor and pcls_net_forward_in16.  ``out`` may hold
  preallocated ``predictions`` / ``probabilities`` for the merged results."""
  if not (torch.is_tensor(raw) and raw.is_cuda and raw.dtype == torch.float32 and raw.dim() == 4 and
          raw.shape[3] in (5, 6)):
    raise ValueError("test-time augmentation needs the RAW input: a float32 CUDA tensor [B,H,W,5|6] (x, y, z, "
                     "remission, range[, label]); the normalised input cannot be mirrored exactly")
  raw = raw.contiguous()
  mc = model.mc
  B, H, W, C = raw.shape
  if (H, W) != (model.ZENITH_LEVEL, model.AZIMUTH_LEVEL):
    raise ValueError("input is %dx%d but the model was built for %dx%d" % (H, W, model.ZENITH_LEVEL, model.AZIMUTH_LEVEL))
  flip, shift, cs, sn = tta.views(W)
  T = len(flip)
  n = T * B
  lib = _lib.load()
  s = stream_handle()
  dev = raw.device
  c_flip, c_shift = _c_array(ctypes.c_int, flip), _c_array(ctypes.c_int, shift)
  mean = _c_array(ctypes.c_double, np.asarray(mc.INPUT_MEAN, np.float64).reshape(-1)[:5])
  std = _c_array(ctypes.c_double, np.asarray(mc.INPUT_STD, np.float64).reshape(-1)[:5])
  out = out or {}
  preds = out.get("predictions")
  if preds is None:
    preds = torch.empty((B, H, W), dtype=torch.int32, device=dev)
  probs = None
  if want_probabilities:
    probs = out.get("probabilities")
    if probs is None:
      probs = torch.empty((B, H, W, mc.NUM_CLASS), dtype=torch.float32, device=dev)
  if n == 0:
    return dict(predictions=preds, **({"probabilities": probs} if probs is not None else {}))
  inp, msk, frames = model.input_buffers(n)
  if frames >= n:
    mask_ptr = msk.value
    _lib.check(lib.pcls_tta_views(ptr(raw), C, B, H, W, mean, std, T, c_flip, c_shift, _c_array(ctypes.c_double, cs),
                                  _c_array(ctypes.c_double, sn), model.precision, inp, msk, s), "pcls_tta_views")
    fwd = model.forward_staged(n, want_probabilities=True)
  else:
    x16 = torch.empty((n, H, W, 8), dtype=torch.float16 if model.precision == _lib.PCLS_F16 else torch.bfloat16,
                      device=dev)
    m = torch.empty((n, H, W), dtype=torch.uint8, device=dev)
    mask_ptr = ptr(m)
    _lib.check(lib.pcls_tta_views(ptr(raw), C, B, H, W, mean, std, T, c_flip, c_shift, _c_array(ctypes.c_double, cs),
                                  _c_array(ctypes.c_double, sn), model.precision, ptr(x16), ptr(m), s), "pcls_tta_views")
    fwd = model.forward_device(x16, m, want_probabilities=True)
  _lib.check(lib.pcls_tta_merge(ptr(fwd["probabilities"]), mask_ptr, B, H, W, mc.NUM_CLASS, mc.CLASSES.index("None"), T,
                                c_flip, c_shift, ptr(probs), ptr(preds), s), "pcls_tta_merge")
  res = {"predictions": preds}
  if probs is not None:
    res["probabilities"] = probs
  return res


def add_tta_flags(parser):
  """``--tta`` / ``--tta_shifts`` of the inference, eval and segment_scans CLIs (see ``from_args``)."""
  parser.add_argument("--tta", action="store_true",
                      help="test-time augmentation: also run the mirror image of every view and average the probabilities")
  parser.add_argument("--tta_shifts", type=str, default=None,
                      help="test-time augmentation: comma-separated column rolls, e.g. 0,1024 (the half turn at W = 2048); "
                           "default 0")
