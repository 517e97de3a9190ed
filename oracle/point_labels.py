"""Per-point labels from range-image predictions: a vectorised numpy restatement of the contract of pcls_point_labels
(include/pclseg.h) - the k-NN vote in a search x search window with neighbours ranked by range difference (the
post-processing published with RangeNet++; parity with RangeNet++'s own code is not claimed).

Inputs are per scan: the per-pixel winner range and prediction, per point its pixel (px, py; -1 = dropped) and range.
Every distance is computed in float32 with separate roundings, the selection is a stable sort on it."""
import numpy as np


def window_weights(search, sigma):
  """1 - g / sum(g), g = exp(-(dx^2 + dy^2) / (2 sigma^2)) over the window, in float64, rounded once to float32."""
  p = (search - 1) // 2
  dy, dx = np.mgrid[-p:p + 1, -p:p + 1].astype(np.float64)
  g = np.exp(-(dx * dx + dy * dy) / (2.0 * float(sigma) ** 2))
  return (1.0 - g / g.sum()).reshape(-1).astype(np.float32)


def point_labels(pred, win_range, valid, px, py, rho, num_classes, none_index, search=1, k=1, weights=None, cutoff=0.0,
                 ignore_class=-1):
  """pred [H,W] int, win_range [H,W] float32 (the winner's range; ignored where ~valid), valid [H,W] bool (pixel not
  empty), px / py [N] int (-1 = dropped point), rho [N] float32 -> [N] int32 labels."""
  H, W = pred.shape
  px, py = np.asarray(px, np.int64), np.asarray(py, np.int64)
  rho = np.asarray(rho, np.float32)
  out = np.full(px.shape[0], none_index, np.int32)
  keep = px >= 0
  if not keep.any():
    return out
  x, y, r = px[keep], py[keep], rho[keep]
  centre = pred[y, x].astype(np.int32)
  if search == 1:
    out[keep] = centre
    return out
  p = (search - 1) // 2
  w = np.ones(search * search, np.float32) if weights is None else np.asarray(weights, np.float32).reshape(-1)
  dy, dx = np.mgrid[-p:p + 1, -p:p + 1]
  dy, dx = dy.reshape(-1), dx.reshape(-1)                      # entry j = (dy+p)*search + (dx+p)
  yy, xx = y[:, None] + dy[None, :], x[:, None] + dx[None, :]  # [n, S*S]
  inside = (yy >= 0) & (yy < H) & (xx >= 0) & (xx < W)
  yc, xc = np.clip(yy, 0, H - 1), np.clip(xx, 0, W - 1)
  ok = inside & valid[yc, xc]
  lab = pred[yc, xc].astype(np.int64)
  rj = win_range[yc, xc].astype(np.float32)
  c = (search * search) // 2
  rj[:, c] = r                                                 # the centre entry uses the point's own range
  lab[:, c] = centre
  ok[:, c] = True
  d = (np.abs(rj - r[:, None]).astype(np.float32) * w[None, :]).astype(np.float32)
  d_sort = np.where(ok, d, np.float32(np.inf))
  order = np.argsort(d_sort, axis=1, kind="stable")            # ties: lower j
  order = np.take_along_axis(order, np.argsort(~np.take_along_axis(ok, order, 1), axis=1, kind="stable"), 1)
  rank = np.empty_like(order)
  np.put_along_axis(rank, order, np.arange(search * search)[None, :].repeat(order.shape[0], 0), 1)
  sel = ok & (rank < k)
  vote = sel & (lab != ignore_class)
  if np.float32(cutoff) > 0:
    vote &= d <= np.float32(cutoff)
  counts = np.stack([(vote & (lab == cls)).sum(1) for cls in range(num_classes)], 1)
  best = counts.argmax(1).astype(np.int32)                     # ties: lowest class
  out[keep] = np.where(counts.max(1) > 0, best, centre)
  return out


def point_labels_batch(pred, win_range, valid, offsets, px, py, rho, num_classes, none_index, **kw):
  """The batched form: pred / win_range / valid [B,H,W], offsets [B+1], per-point arrays over the whole batch."""
  out = np.empty(int(offsets[-1]), np.int32)
  for b in range(pred.shape[0]):
    lo, hi = int(offsets[b]), int(offsets[b + 1])
    out[lo:hi] = point_labels(pred[b], win_range[b], valid[b], px[lo:hi], py[lo:hi], rho[lo:hi], num_classes,
                              none_index, **kw)
  return out


def winner_range(keys, offsets, unproj_range):
  """The per-pixel winner range and validity from the scatter's keys [B,H,W] (int64 bit patterns, -1 = empty): the
  range is read through the key's low word (the winner's local index), for both projection variants."""
  keys = np.asarray(keys).view(np.uint64)
  valid = keys != np.uint64(0xFFFFFFFFFFFFFFFF)
  idx = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64) + np.asarray(offsets[:-1], np.int64)[:, None, None]
  rng = np.zeros(keys.shape, np.float32)
  rng[valid] = np.asarray(unproj_range, np.float32)[idx[valid]]
  return rng, valid
