"""Monte-Carlo (MC) dropout on the GPU: epistemic uncertainty from T stochastic forward passes with the network's Dropout
layers active (Gal & Ghahramani, ICML 2016; Kendall et al., Bayesian SegNet, 2015).  Per pixel: the mean probabilities
and their argmax, the predictive entropy H of the mean and the mutual information MI = H - E_t[h_t] between prediction and
weights.  ``pcls_confidence`` reports the spread of ONE softmax (aleatoric); MI is large where the passes disagree, i.e.
where the weights are unsure.

The stochastic net is a second pcls_net handle (``model.mc_net``), built on first use: the default net, its call sequence
and its outputs are not touched.  The dropout mask of an element depends only on (seed, global frame id, pass, site), so
results do not depend on the batch, the micro batch, graph replay or the number of GPUs.  The rules are in
include/pclseg.h and oracle/mc_dropout.py.  No claim is made about the quality of the uncertainty on trained weights."""
import ctypes

import numpy as np
import torch

from . import _lib
from .calibration import raw_mask
from .device import ptr, stream_handle

MAX_PASSES = 256


def dropout_threshold(rate):
  """thr = floor(rate * 65536 + 0.5) in float64 (the kernels' keep rule: u16 >= thr)."""
  return int(np.floor(float(rate) * 65536.0 + 0.5))


def check_rate(rate):
  rate = float(rate)
  if not (np.isfinite(rate) and rate >= 0.0 and dropout_threshold(rate) < 65536):
    raise ValueError("dropout rate must be finite, >= 0 and below 1 - 2^-17, got %r" % rate)
  return rate


class MCDropout:
  """``passes`` T stochastic forward passes (1 .. 256) with the Dropout layers active at ``rate`` (None: the config's
  ``DROP_RATE``), masks drawn from ``seed`` (0 <= seed < 2^64).  ``next_frame`` is the global id of the next frame a
  call sees; each call advances it by its batch, so consecutive batches get different masks.  Set it to the first
  global frame index of a shard to reproduce the single-GPU masks on several GPUs."""

  def __init__(self, passes=8, seed=0, rate=None):
    self.passes, self.seed = int(passes), int(seed)
    self.rate = None if rate is None else float(rate)
    self.next_frame = 0
    if not 1 <= self.passes <= MAX_PASSES:
      raise ValueError("passes must be in [1, %d], got %d" % (MAX_PASSES, self.passes))
    if not 0 <= self.seed < 1 << 64:
      raise ValueError("seed must be in [0, 2^64), got %d" % self.seed)
    if self.rate is not None:
      check_rate(self.rate)

  def rate_for(self, mc):
    """The dropout rate used with config ``mc``."""
    return check_rate(self.rate if self.rate is not None else float(mc.DROP_RATE))

  def __repr__(self):
    return "MCDropout(passes=%d, seed=%d, rate=%r)" % (self.passes, self.seed, self.rate)


def check_exclusive(mcd, tta=None, calibration=None):
  """MC dropout is not combined with test-time augmentation or with a softmax temperature / fit."""
  if mcd is None:
    return
  if tta is not None:
    raise ValueError("MC dropout cannot be combined with test-time augmentation")
  if calibration is not None and (calibration.temperature != 1.0 or calibration.fit):
    raise ValueError("MC dropout cannot be combined with a softmax temperature or a temperature fit: its confidence "
                     "is the max of the mean probabilities")


def accumulate(probs, n_pass, acc_probs, acc_entropy, num_classes):
  """pcls_mc_accumulate: probs [..., NC] float32 CUDA of pass ``n_pass`` into acc_probs / acc_entropy (in place)."""
  _lib.check(_lib.load().pcls_mc_accumulate(ptr(probs), acc_entropy.numel(), int(num_classes), int(n_pass),
                                            ptr(acc_probs), ptr(acc_entropy), stream_handle()), "pcls_mc_accumulate")


def finalize(acc_probs, acc_entropy, mask, num_classes, none_index, passes, want_probabilities=True, out=None):
  """pcls_mc_finalize -> dict(predictions, confidence, entropy, mutual_information, probabilities?) of the shape of
  ``acc_entropy`` (``mask``: uint8 CUDA tensor, a device pointer, or None = all valid)."""
  shape = tuple(acc_entropy.shape)
  dev = acc_entropy.device
  out = out or {}
  res = {"predictions": out.get("predictions")}
  if res["predictions"] is None:
    res["predictions"] = torch.empty(shape, dtype=torch.int32, device=dev)
  for k in ("confidence", "entropy", "mutual_information"):
    res[k] = torch.empty(shape, dtype=torch.float32, device=dev)
  if want_probabilities:
    res["probabilities"] = out.get("probabilities")
    if res["probabilities"] is None:
      res["probabilities"] = torch.empty(shape + (int(num_classes),), dtype=torch.float32, device=dev)
  mask_ptr = mask if isinstance(mask, ctypes.c_void_p) else ptr(mask)
  _lib.check(_lib.load().pcls_mc_finalize(ptr(acc_probs), ptr(acc_entropy), mask_ptr, acc_entropy.numel(),
                                          int(num_classes), int(none_index), int(passes),
                                          ptr(res.get("probabilities")), ptr(res["predictions"]),
                                          ptr(res["confidence"]), ptr(res["entropy"]),
                                          ptr(res["mutual_information"]), stream_handle()), "pcls_mc_finalize")
  return res


def forward_mc(model, raw, mcd, want_probabilities=False, out=None):
  """T stochastic passes over one batch -> dict(predictions [B,H,W] int32, confidence / entropy / mutual_information
  [B,H,W] float32, probabilities [B,H,W,NC] float32 when asked), all CUDA.

  ``raw``: float32 CUDA RAW range images [B,H,W,5|6] (x, y, z, remission, range[, label]).  The staged network input is
  released by liveness after its last reader, so every pass stages it again through pcls_net_forward's raw input path.
  Frames get the global ids ``mcd.next_frame`` .. ``+ B - 1``; the counter then advances by B."""
  if not (torch.is_tensor(raw) and raw.is_cuda and raw.dtype == torch.float32 and raw.dim() == 4 and
          raw.shape[3] in (5, 6)):
    raise ValueError("MC dropout needs float32 CUDA RAW range images [B,H,W,5|6] (x, y, z, remission, range[, label])")
  mc = model.mc
  B, H, W, C = raw.shape
  if (H, W) != (model.ZENITH_LEVEL, model.AZIMUTH_LEVEL):
    raise ValueError("input is %dx%d but the model was built for %dx%d" % (H, W, model.ZENITH_LEVEL,
                                                                          model.AZIMUTH_LEVEL))
  raw = raw.contiguous()
  nc, none = mc.NUM_CLASS, mc.CLASSES.index("None")
  lib = _lib.load()
  s = stream_handle()
  dev = raw.device
  net = model.mc_net(mcd.rate_for(mc), B)
  preds_t = torch.empty((B, H, W), dtype=torch.int32, device=dev)
  probs_t = torch.empty((B, H, W, nc), dtype=torch.float32, device=dev)
  acc_p = torch.empty((B, H, W, nc), dtype=torch.float32, device=dev)
  acc_h = torch.empty((B, H, W), dtype=torch.float64, device=dev)
  m = raw_mask(raw, mc)
  mean = (ctypes.c_double * 5)(*np.asarray(mc.INPUT_MEAN, np.float64).reshape(-1)[:5])
  std = (ctypes.c_double * 5)(*np.asarray(mc.INPUT_STD, np.float64).reshape(-1)[:5])
  frame_base = mcd.next_frame
  for t in range(mcd.passes if B else 0):
    _lib.check(lib.pcls_net_set_dropout(net, mcd.seed, frame_base, t, s), "pcls_net_set_dropout")
    _lib.check(lib.pcls_net_forward(net, ptr(raw), C, None, mean, std, B, None, ptr(probs_t), ptr(preds_t), s),
               "pcls_net_forward")
    accumulate(probs_t, t, acc_p, acc_h, nc)
  mcd.next_frame = frame_base + B
  return finalize(acc_p, acc_h, m, nc, none, mcd.passes, want_probabilities=want_probabilities, out=out)


def add_mc_flags(parser):
  """``--mc_dropout T [--mc_seed S] [--mc_rate r]`` of the inference, eval and segment_scans CLIs."""
  parser.add_argument("--mc_dropout", type=int, default=None, metavar="T",
                      help="Monte-Carlo dropout: T stochastic forward passes; reports the predictive entropy and the "
                           "mutual information")
  parser.add_argument("--mc_seed", type=int, default=0, help="Monte-Carlo dropout: seed of the dropout masks")
  parser.add_argument("--mc_rate", type=float, default=None,
                      help="Monte-Carlo dropout: dropout rate (default: the config's DROP_RATE)")


def from_args(args):
  """The CLIs' MC flags: None (the plain path) without ``--mc_dropout``."""
  if getattr(args, "mc_dropout", None) is None:
    return None
  return MCDropout(passes=args.mc_dropout, seed=args.mc_seed, rate=args.mc_rate)
