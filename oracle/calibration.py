"""numpy restatement of the calibration contract (include/pclseg.h: pcls_confidence, pcls_temperature_nll,
pcls_reliability_update, pcls_point_confidence) in float64, the bin rule with a float32 product, ECE / MCE and the
temperature fit (a parabola through log T at the grid's argmin)."""
import numpy as np

U = 2.0 ** -24   # float32 unit roundoff


def inv_temperature(T):
  return np.float32(1.0 / float(T))


def softmax(z, a):
  """softmax(z * a) over the last axis in float64 from float32 z and float32 a."""
  s = np.asarray(z, np.float64) * np.float64(a)
  s = s - s.max(-1, keepdims=True)
  e = np.exp(s)
  return e / e.sum(-1, keepdims=True)


def confidence(logits=None, probs=None, mask=None, a=np.float32(1.0)):
  """(probs, conf, entropy) in float64: conf = max_c p_c, entropy = -sum p log p / log NC (0 for NC = 1), both 0 where
  mask == 0."""
  p = softmax(logits, a) if logits is not None else np.asarray(probs, np.float64)
  nc = p.shape[-1]
  conf = p.max(-1)
  with np.errstate(divide="ignore", invalid="ignore"):
    plogp = np.where(p > 0, p * np.log(np.where(p > 0, p, 1.0)), 0.0)
  ent = -plogp.sum(-1) / np.log(nc) if nc > 1 else np.zeros(conf.shape)
  if mask is not None:
    valid = np.asarray(mask) != 0
    conf, ent = np.where(valid, conf, 0.0), np.where(valid, ent, 0.0)
  return p, conf, ent


def counted(label, nc, ignore_index):
  label = np.asarray(label, np.int64)
  return (label >= 0) & (label < nc) & (label != ignore_index)


def temperature_nll(logits, label, nc, ignore_index, inv_temps):
  """(sums [n_temps] float64, count, bound [n_temps]): the float64 value of the kernel's float32 expression
  term = (log sum_c exp(s_c - m) + m) - s_label, s = z * a_t, summed over the counted pixels, and a bound on how far the
  float32 evaluation may be from it.  Per term, with S = max_c |s_c| and u = 2^-24: s_c and m carry u S, s_c - m 4 u S,
  expf (<= 2 ulp) 4 u relative, the NC-term float32 sum NC u relative, logf 1 ulp of |log e| <= log NC, then + m and
  - s_label two roundings of values <= 2 S + log NC and u S each from the inputs: |err| <= u (10 S + NC + 3 log NC + 8);
  the bound is that summed over the counted pixels (float64 accumulation adds far less)."""
  z = np.asarray(logits, np.float32).reshape(-1, nc)
  y = np.asarray(label).reshape(-1)
  ok = counted(y, nc, ignore_index)
  z, y = z[ok].astype(np.float64), y[ok].astype(np.int64)
  sums, bound = [], []
  for a in inv_temps:
    s = z * np.float64(np.float32(a))
    m = s.max(1)
    term = np.log(np.exp(s - m[:, None]).sum(1)) + m - s[np.arange(y.size), y]
    S = np.abs(s).max(1) if y.size else np.zeros(0)
    sums.append(term.sum())
    bound.append((U * (10 * S + nc + 3 * np.log(nc) + 8)).sum())
  return np.array(sums), int(ok.sum()), np.array(bound)


def bin_index(conf, n_bins):
  """b = min((int)(conf * (float)n_bins), n_bins - 1), the product rounded to float32, clamped at 0."""
  prod = np.asarray(conf, np.float32) * np.float32(n_bins)
  return np.clip(np.trunc(prod), 0, n_bins - 1).astype(np.int64)


def reliability(conf, pred, label, nc, ignore_index, n_bins):
  """(count int64 [n_bins], correct int64 [n_bins], conf_sum float64 [n_bins])."""
  conf = np.asarray(conf, np.float32).reshape(-1)
  pred = np.asarray(pred, np.int64).reshape(-1)
  label = np.asarray(label, np.int64).reshape(-1)
  ok = counted(label, nc, ignore_index) & (pred >= 0) & (pred < nc)
  b = bin_index(conf[ok], n_bins)
  count = np.bincount(b, minlength=n_bins).astype(np.int64)
  correct = np.bincount(b, weights=(pred[ok] == label[ok]), minlength=n_bins).astype(np.int64)
  conf_sum = np.bincount(b, weights=conf[ok].astype(np.float64), minlength=n_bins)
  return count, correct, conf_sum


def ece_mce(count, correct, conf_sum):
  """ECE = sum_b |correct_b - conf_b| / N and MCE = max over non-empty bins of |acc_b - conf_b|."""
  count = np.asarray(count, np.float64)
  n = count.sum()
  if n == 0:
    return 0.0, 0.0
  full = count > 0
  ece = np.abs(np.asarray(correct, np.float64) - conf_sum).sum() / n
  mce = np.abs(np.asarray(correct, np.float64)[full] / count[full] - np.asarray(conf_sum)[full] / count[full]).max()
  return float(ece), float(mce)


def point_confidence(probs, offsets, proj_x, proj_y, point_labels):
  """out[i] = probs[b, proj_y[i], proj_x[i], label[i]]; 0 for proj_x < 0 or a label outside [0, NC)."""
  nc = probs.shape[-1]
  total = proj_x.size
  scan = np.searchsorted(np.asarray(offsets), np.arange(total), side="right") - 1
  ok = (proj_x >= 0) & (point_labels >= 0) & (point_labels < nc)
  out = np.zeros(total, np.float32)
  out[ok] = probs[scan[ok], proj_y[ok], proj_x[ok], point_labels[ok]]
  return out


def log_grid(lo, hi, points):
  t = np.exp(np.linspace(np.log(lo), np.log(hi), points))
  t[0], t[-1] = lo, hi
  return t


def fit(temps, nll):
  """(t_star, at_edge): exp of the vertex of the parabola through (log T, NLL) at the argmin and its neighbours
  (np.polyfit), or the grid end with at_edge."""
  k = int(np.argmin(nll))
  if k in (0, len(temps) - 1):
    return float(temps[k]), True
  x = np.log(np.asarray(temps[k - 1:k + 2], np.float64))
  c2, c1, _ = np.polyfit(x, np.asarray(nll[k - 1:k + 2], np.float64), 2)
  return float(np.exp(-c1 / (2 * c2))), False
