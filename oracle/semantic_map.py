"""Semantic map fusion in numpy (the rules of pcls_semantic_map_vote / _query in include/pclseg.h): float64 voxel keys
computed in the kernels' operation order (numpy rounds every product and sum on its own), vote counts from np.unique,
and the relabel and export rules.  The GPU is compared against this bit for bit."""
import numpy as np

HALF = 1 << 20           # voxel indices in [-2^20, 2^20)


def pose_rows(poses):
  """[B,4,4] or [B,3,4] or [B,12] -> [B,12] float64 (the 3x4 row-major (R | t))."""
  p = np.asarray(poses, np.float64)
  if p.ndim == 3:
    p = p[:, :3, :]
  return p.reshape(-1, 12)


def voxel_keys(points, offsets, poses, voxel_size):
  """points [total,>=3] float32, offsets [B+1], poses [B,...] -> (keys [total] uint64, has_voxel [total] bool).  Keys of
  points without a voxel are 0."""
  pts = np.asarray(points, np.float32)
  x, y, z = (pts[:, k].astype(np.float64) for k in range(3))
  rows = pose_rows(poses)
  offsets = np.asarray(offsets, np.int64)
  scan = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets))
  r = rows[scan]
  s = np.float64(voxel_size)
  ok = np.ones(pts.shape[0], bool)
  v = []
  with np.errstate(invalid="ignore", over="ignore"):
    for k in range(3):
      w = ((r[:, 4 * k] * x + r[:, 4 * k + 1] * y) + r[:, 4 * k + 2] * z) + r[:, 4 * k + 3]
      f = np.floor(w / s)
      ok &= np.isfinite(w) & (f >= -HALF) & (f < HALF)
      v.append(f)
  keys = np.zeros(pts.shape[0], np.uint64)
  for k, f in enumerate(v):
    idx = np.where(ok, f, 0).astype(np.int64) + HALF
    keys |= idx.astype(np.uint64) << np.uint64(42 - 21 * k)
  keys[~ok] = 0
  return keys, ok


def pack_key(vx, vy, vz):
  return np.uint64(((int(vx) + HALF) << 42) | ((int(vy) + HALF) << 21) | (int(vz) + HALF))


def unpack_keys(keys):
  """uint64 keys -> [V,3] int32 voxel indices."""
  k = np.asarray(keys, np.uint64)
  m = np.uint64((1 << 21) - 1)
  return np.stack([((k >> np.uint64(s)) & m).astype(np.int64) - HALF for s in (42, 21, 0)], 1).astype(np.int32)


def voters(points, offsets, poses, voxel_size, labels, num_classes, ignore_class=-1, min_range=0.0, max_range=0.0):
  """The votes of one call: (keys, labels) of the points that vote."""
  pts = np.asarray(points, np.float32)
  labels = np.asarray(labels).astype(np.int64)
  keys, ok = voxel_keys(pts, offsets, poses, voxel_size)
  x, y, z = (pts[:, k].astype(np.float64) for k in range(3))
  r2 = (x * x + y * y) + z * z
  ok &= (labels >= 0) & (labels < num_classes) & (labels != ignore_class)
  with np.errstate(invalid="ignore"):
    ok &= r2 >= np.float64(min_range) * np.float64(min_range)
    if max_range > 0:
      ok &= r2 <= np.float64(max_range) * np.float64(max_range)
  return keys[ok], labels[ok]


def table(vote_keys, vote_labels, num_classes):
  """All votes -> (keys [V] uint64 ascending, counts [V,NC] uint32)."""
  keys, inv = np.unique(np.asarray(vote_keys, np.uint64), return_inverse=True)
  counts = np.zeros((keys.size, num_classes), np.uint32)
  np.add.at(counts, (inv.reshape(-1), np.asarray(vote_labels, np.int64)), 1)
  return keys, counts


def export(keys, counts, voxel_size):
  """The map as ``SemanticMap.export()`` returns it: sorted by key, labels = argmax (ties to the lowest class)."""
  return dict(voxels=unpack_keys(keys), counts=np.asarray(counts, np.uint32),
              labels=np.argmax(counts, axis=1).astype(np.int32) if len(keys) else np.zeros(0, np.int32),
              voxel_size=np.float64(voxel_size))


def relabel(points, offsets, poses, voxel_size, labels_in, keys, counts, keep_mask=0, min_votes=1):
  """pcls_semantic_map_query: [total] int32."""
  labels_in = np.asarray(labels_in).astype(np.int32)
  out = labels_in.copy()
  pk, ok = voxel_keys(points, offsets, poses, voxel_size)
  keep = (labels_in >= 0) & (labels_in < 32) & ((np.uint64(keep_mask) >> np.clip(labels_in, 0, 31).astype(np.uint64))
                                               & np.uint64(1)).astype(bool)
  if len(keys) == 0:
    return out
  pos = np.clip(np.searchsorted(keys, pk), 0, len(keys) - 1)
  found = ok & (keys[pos] == pk)
  total = counts.astype(np.int64).sum(1)
  take = found & ~keep & (total[pos] >= min_votes)
  out[take] = np.argmax(counts[pos[take]], axis=1)
  return out
