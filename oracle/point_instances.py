"""Instance ids for thing-class points: a vectorised numpy restatement of the contract of pcls_point_instances
(include/pclseg.h) - connected components in the range image.  Bit parity with any published clustering code is not
claimed.

Per scan b, with the winner keys of pcls_project_scatter (the low word is the winner's local index) and per-point labels L:
1. A node is a pixel (r, c) whose winner i has L[i] in the thing set (a uint32 bitmask over classes).
2. Nodes u, v are joined when |r_u - r_v| <= ry, the column distance is <= rx (taken modulo W with wrap, so that columns
   0 and W-1 are neighbours), L is equal at both and d^2 <= tau^2: d^2 = (dx*dx + dy*dy) + dz*dz in float32 with separate
   roundings over the two winners' x, y, z, tau^2 = fl32(tau * tau).
3. Components are the connected components of that graph.
4. A node's winner belongs to its component.  A non-winner point j at a node's pixel belongs to it when L[j] equals the
   winner's label and d^2(j, winner) <= tau^2.  Every other point (stuff classes, dropped points, occluded points that
   fail the test) belongs to no component.
5. A component's size is the number of points that belong to it.  Components with size >= min_points are numbered 1, 2,
   ... per scan in increasing order of their smallest pixel index r*W + c; every other point gets 0.
"""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)


def dist2(a, b):
  """[..., 3] float32 pairs -> d^2 in float32, (dx*dx + dy*dy) + dz*dz with separate roundings."""
  a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
  d = (a - b).astype(np.float32)
  sq = (d * d).astype(np.float32)
  return ((sq[..., 0] + sq[..., 1]).astype(np.float32) + sq[..., 2]).astype(np.float32)


def forward_window(ry, rx):
  """The forward half of the (2 ry + 1) x (2 rx + 1) window: every unordered pair of pixels once."""
  return [(dr, dc) for dr in range(0, ry + 1) for dc in range(-rx, rx + 1) if dr > 0 or dc > 0]


def scan_instances(points, keys, px, py, labels, thing_mask, ry, rx, wrap, tau, min_points):
  """One scan: points [N,>=3] float32, keys [H,W] (uint64 bit patterns, ~0 = empty; low word = local winner index),
  px / py [N] (-1 = dropped), labels [N] int -> (instances [N] int32, count, stats dict(nodes, edges_tested, edges))."""
  keys = np.asarray(keys).view(np.uint64)
  H, W = keys.shape
  pts = np.asarray(points, np.float32)[:, :3]
  labels = np.asarray(labels, np.int64)
  px, py = np.asarray(px, np.int64), np.asarray(py, np.int64)
  n_pts = pts.shape[0]
  tau2 = np.float32(np.float32(tau) * np.float32(tau))
  occupied = keys != EMPTY
  win = np.where(occupied, (keys & np.uint64(0xFFFFFFFF)).astype(np.int64), -1)
  wl = np.where(occupied, labels[np.maximum(win, 0)] if n_pts else 0, -1)
  is_thing = (wl >= 0) & (wl < 32) & ((np.uint64(thing_mask) >> np.clip(wl, 0, 31).astype(np.uint64)) & np.uint64(1)
                                      ).astype(bool)
  node = occupied & is_thing
  xyz = np.zeros((H, W, 3), np.float32)
  if n_pts:
    xyz[occupied] = pts[win[occupied]]
  pix = np.arange(H * W).reshape(H, W)
  src, dst = [], []
  tested = 0
  for dr, dc in forward_window(ry, rx):
    r0 = np.arange(H - dr)
    c0 = np.arange(W)
    c1 = c0 + dc
    if wrap:
      c1 = c1 % W
      cs = np.ones(W, bool)
    else:
      cs = (c1 >= 0) & (c1 < W)
    c0, c1 = c0[cs], c1[cs]
    a = (r0[:, None], c0[None, :])
    b = (r0[:, None] + dr, c1[None, :])
    both = node[a] & node[b]
    tested += int(both.sum())
    ok = both & (wl[a] == wl[b]) & (dist2(xyz[a], xyz[b]) <= tau2)
    src.append(pix[a][ok])
    dst.append(pix[b][ok])
  src = np.concatenate(src) if src else np.zeros(0, np.int64)
  dst = np.concatenate(dst) if dst else np.zeros(0, np.int64)
  g = coo_matrix((np.ones(src.size, np.int8), (src, dst)), shape=(H * W, H * W))
  _, comp = connected_components(g, directed=False)
  flat_node = node.reshape(-1)
  # root of a component = its smallest pixel index
  root_of_comp = np.full(H * W, H * W, np.int64)
  np.minimum.at(root_of_comp, comp[flat_node], pix.reshape(-1)[flat_node])
  root = np.where(flat_node, root_of_comp[comp], -1)
  # rule 4
  belongs = np.full(n_pts, -1, np.int64)
  keep = px >= 0
  idx = np.flatnonzero(keep)
  p = py[idx] * W + px[idx]
  rp = root[p]
  w = win.reshape(-1)[p]
  at_node = rp >= 0
  same = idx == w
  test = at_node & ~same
  ok = np.zeros(idx.size, bool)
  if test.any():
    ok[test] = (labels[idx[test]] == labels[w[test]]) & (dist2(pts[idx[test]], pts[w[test]]) <= tau2)
  inn = at_node & (same | ok)
  belongs[idx[inn]] = rp[inn]
  size = np.bincount(belongs[belongs >= 0], minlength=H * W)
  kept_roots = np.flatnonzero(size >= min_points)            # increasing pixel index
  ids = np.zeros(H * W, np.int32)
  ids[kept_roots] = np.arange(1, kept_roots.size + 1, dtype=np.int32)
  out = np.where(belongs >= 0, ids[np.maximum(belongs, 0)], 0).astype(np.int32)
  return out, int(kept_roots.size), dict(nodes=int(node.sum()), edges_tested=tested, edges=int(src.size))


def point_instances(points, keys, offsets, px, py, labels, thing_mask, ry=1, rx=2, wrap=True, tau=0.5, min_points=10):
  """The batched form: points [total,4], keys [B,H,W], offsets [B+1], per-point arrays over the whole batch ->
  (instances [total] int32, counts [B] int32)."""
  offsets = np.asarray(offsets, np.int64)
  B = offsets.shape[0] - 1
  out = np.zeros(int(offsets[-1]), np.int32)
  counts = np.zeros(B, np.int32)
  for b in range(B):
    lo, hi = int(offsets[b]), int(offsets[b + 1])
    out[lo:hi], counts[b], _ = scan_instances(points[lo:hi], keys[b], px[lo:hi], py[lo:hi], labels[lo:hi], thing_mask,
                                              ry, rx, wrap, tau, min_points)
  return out, counts


def keys_from_pixels(px, py, rng_val, offsets, H, W):
  """Winner keys [B,H,W] (int64 bit patterns) from per-point pixels and ranges by the scatter's rule (nearest point,
  then lowest index) - for hand-built cases that do not run the projection."""
  offsets = np.asarray(offsets, np.int64)
  B = offsets.shape[0] - 1
  keys = np.full((B, H, W), EMPTY, np.uint64)
  r = np.asarray(rng_val, np.float32)
  for b in range(B):
    for i in range(int(offsets[b]), int(offsets[b + 1])):
      if px[i] < 0:
        continue
      k = (np.uint64(r[i:i + 1].view(np.uint32)[0]) << np.uint64(32)) | np.uint64(i - offsets[b])
      keys[b, py[i], px[i]] = min(keys[b, py[i], px[i]], k)
  return keys.view(np.int64)
