"""Calibrated confidence on the GPU: post-hoc temperature scaling (Guo et al., "On Calibration of Modern Neural
Networks", ICML 2017).  One scalar T is fitted on a validation set by minimising the NLL of softmax(z / T) over a
log-spaced grid (pcls_temperature_nll evaluates up to 64 temperatures per pass over the logits); confidences are computed
at T (pcls_confidence) and their reliability is measured with ``metrics.Reliability`` (ECE / MCE).  The argmax does not
depend on T, so the predictions stay what they are.  The kernel rules are in include/pclseg.h and oracle/calibration.py.
"""
import ctypes
import math

import numpy as np
import torch

from . import _lib
from .device import ptr, stream_handle

MAX_TEMPS = 64   # temperatures per pcls_temperature_nll pass
MAX_BINS = 64


def inv_temperature(T):
  """a = 1 / T computed in float64 and rounded once to float32 (the kernels' argument)."""
  return float(np.float32(1.0 / float(T)))


class Calibration:
  """What to compute about confidence: the working ``temperature`` T (> 0; confidences are max softmax(z / T)),
  ``n_bins`` equal reliability bins of [0, 1] (1 .. 64), and with ``fit`` the NLL over ``grid = (lo, hi, points)``:
  ``points`` (2 .. 64) log-spaced temperatures from lo to hi, both ends included."""

  def __init__(self, temperature=1.0, n_bins=15, fit=False, grid=(0.25, 4.0, 64)):
    self.temperature, self.n_bins, self.fit = float(temperature), int(n_bins), bool(fit)
    lo, hi, points = float(grid[0]), float(grid[1]), int(grid[2])
    self.grid = (lo, hi, points)
    if not (math.isfinite(self.temperature) and self.temperature > 0):
      raise ValueError("temperature must be finite and > 0, got %r" % (temperature,))
    if not 1 <= self.n_bins <= MAX_BINS:
      raise ValueError("n_bins must be in [1, %d], got %d" % (MAX_BINS, self.n_bins))
    if not 2 <= points <= MAX_TEMPS:
      raise ValueError("the grid needs 2 .. %d points, got %d" % (MAX_TEMPS, points))
    if not (math.isfinite(lo) and math.isfinite(hi) and 0 < lo < hi):
      raise ValueError("the grid needs 0 < lo < hi, got (%r, %r)" % (lo, hi))

  def grid_temperatures(self):
    """The fit's grid: float64 [points], log-spaced, exactly lo and hi at the ends."""
    lo, hi, points = self.grid
    t = np.exp(np.linspace(math.log(lo), math.log(hi), points))
    t[0], t[-1] = lo, hi
    return t

  def __repr__(self):
    return "Calibration(temperature=%r, n_bins=%d, fit=%s, grid=%s)" % (self.temperature, self.n_bins, self.fit,
                                                                        self.grid)


def check_tta(calibration, tta):
  """TTA merges probabilities, not logits: with a TTA only the merged probabilities at T = 1 are available."""
  if calibration is not None and tta is not None and (calibration.temperature != 1.0 or calibration.fit):
    raise ValueError("test-time augmentation merges probabilities, not logits: confidence with TTA is only available at "
                     "temperature 1 and without a temperature fit")


def fit_temperature(temps, nll):
  """(t_star, at_edge) from the NLL on a grid of increasing temperatures: the argmin, refined to exp of the vertex of
  the parabola through (log T, NLL) at the argmin and its two neighbours; at a grid end, that end with at_edge=True."""
  t = np.asarray(temps, np.float64)
  y = np.asarray(nll, np.float64)
  k = int(np.argmin(y))
  if k == 0 or k == t.size - 1:
    return float(t[k]), True
  x0, x1, x2 = np.log(t[k - 1:k + 2])
  y0, y1, y2 = y[k - 1:k + 2]
  den = (x1 - x0) * (y1 - y2) - (x1 - x2) * (y1 - y0)
  if den == 0:
    return float(t[k]), False
  xv = x1 - 0.5 * ((x1 - x0) ** 2 * (y1 - y2) - (x1 - x2) ** 2 * (y1 - y0)) / den
  return float(math.exp(xv)), False


class TemperatureNLL:
  """Device accumulators of pcls_temperature_nll: the summed NLL of softmax(z / T) for the fit's grid (when
  ``calibration.fit``) and for T = 1 and the working temperature, and the number of counted pixels (0 <= label < NC,
  label != ignore_index)."""

  def __init__(self, calibration, num_classes, ignore_index):
    self.calibration, self.num_classes, self.ignore_index = calibration, int(num_classes), int(ignore_index)
    self.grid = calibration.grid_temperatures() if calibration.fit else np.zeros(0)
    self.temps = np.concatenate([self.grid, [1.0, calibration.temperature]])
    self._inv = [(ctypes.c_float * len(c))(*[inv_temperature(T) for T in c])
                 for c in (self.temps[i:i + MAX_TEMPS] for i in range(0, self.temps.size, MAX_TEMPS))]
    self._sum = self._count = None

  def _ensure(self, dev):
    if self._sum is None:
      self._sum = torch.zeros(self.temps.size, dtype=torch.float64, device=dev)
      self._count = torch.zeros(1, dtype=torch.int64, device=dev)

  def update(self, logits, label):
    """logits [..., NC] float32 CUDA, label [...] int32 CUDA (same leading shape)."""
    self._ensure(logits.device)
    n = int(label.numel())
    if logits.numel() != n * self.num_classes:
      raise ValueError("logits hold %d values, label %d pixels x %d classes" % (logits.numel(), n, self.num_classes))
    lib, s, lo = _lib.load(), stream_handle(), 0
    for i, inv in enumerate(self._inv):
      # the pixel count is taken once: every chunk counts the same pixels
      cnt = self._count if i == 0 else torch.zeros(1, dtype=torch.int64, device=logits.device)
      _lib.check(lib.pcls_temperature_nll(ptr(logits), ptr(label), n, self.num_classes, self.ignore_index, len(inv), inv,
                                          ptr(self._sum[lo:lo + len(inv)]), ptr(cnt), s), "pcls_temperature_nll")
      lo += len(inv)

  def allreduce(self, comm):
    """Sums the accumulators over the ranks of ``comm`` (torch.distributed, off the hot path)."""
    self._ensure(torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else "cpu")
    comm.allreduce_sums([self._sum, self._count])

  def result(self):
    """dict(temperatures (the grid), nll (mean NLL per grid temperature), t_star, at_edge (None / False without a fit),
    nll_at_1, nll_at_temperature, counted)."""
    if self._sum is None:
      sums, count = np.zeros(self.temps.size), 0
    else:
      sums, count = self._sum.cpu().numpy(), int(self._count.item())
    mean = sums / count if count else np.full(self.temps.size, np.nan)
    g = self.grid.size
    t_star = at_edge = None
    if g and count:
      t_star, at_edge = fit_temperature(self.grid, mean[:g])
    return dict(temperatures=self.grid.copy(), nll=mean[:g], t_star=t_star, at_edge=at_edge, nll_at_1=float(mean[g]),
                nll_at_temperature=float(mean[g + 1]), temperature=self.calibration.temperature, counted=count)


def confidence(num_classes, logits=None, probs=None, mask=None, temperature=1.0, want_probs=False, want_entropy=False):
  """pcls_confidence over [..., NC] float32 CUDA logits (at ``temperature``) or probabilities (T = 1 only) ->
  dict(confidence [...], probabilities [..., NC]? (with want_probs), entropy [...]? (with want_entropy)); ``mask``
  [...] uint8 CUDA (a tensor or a device pointer) or None (= all valid) zeroes confidence and entropy at empty pixels."""
  src = logits if logits is not None else probs
  shape = tuple(src.shape[:-1])
  n = int(np.prod(shape)) if shape else 1
  dev = src.device
  conf = torch.empty(shape, dtype=torch.float32, device=dev)
  out = {"confidence": conf}
  if want_probs:
    out["probabilities"] = torch.empty(tuple(src.shape), dtype=torch.float32, device=dev)
  if want_entropy:
    out["entropy"] = torch.empty(shape, dtype=torch.float32, device=dev)
  mask_ptr = mask if isinstance(mask, ctypes.c_void_p) else ptr(mask)
  _lib.check(_lib.load().pcls_confidence(ptr(logits), ptr(probs), mask_ptr, n, int(num_classes),
                                         inv_temperature(temperature), ptr(out.get("probabilities")), ptr(conf),
                                         ptr(out.get("entropy")), stream_handle()), "pcls_confidence")
  return out


def raw_mask(frames, mc):
  """uint8 [B,H,W] CUDA mask (range > 0) of raw [B,H,W,5|6] float32 CUDA frames, from the input stage kernel."""
  B, H, W, C = frames.shape
  mask = torch.empty((B, H, W), dtype=torch.uint8, device=frames.device)
  mean = (ctypes.c_double * 5)(*np.asarray(mc.INPUT_MEAN, np.float64).reshape(-1)[:5])
  std = (ctypes.c_double * 5)(*np.asarray(mc.INPUT_STD, np.float64).reshape(-1)[:5])
  _lib.check(_lib.load().pcls_input_stage(ptr(frames), C, B * H * W, mean, std, mc.CLASSES.index("None"), None,
                                          ptr(mask), None, None, 0, None, stream_handle()), "pcls_input_stage")
  return mask


def add_temperature_flag(parser):
  parser.add_argument("--temperature", type=float, default=1.0,
                      help="softmax temperature T of the confidences: max softmax(logits / T) (default 1)")
