"""Semantic map fusion on the GPU: the point labels of a pose-registered sequence voted into a voxel hash map
(pcls_semantic_map_vote), and every point relabelled from the map (pcls_semantic_map_query).  The same wall, road or
parked car is seen in dozens of scans of a sequence; voting per voxel makes the labels of the static scene consistent,
gives points the projection dropped a label, and leaves a labelled map as a by-product.  The voxel, vote and query rules
are in include/pclseg.h and oracle/semantic_map.py.

    m = SemanticMap(num_classes=20, ignore_class=0)
    for batch in sequence:                               # pass 1: vote
      m.vote(points, offsets, poses, point_labels)
    for batch in sequence:                               # pass 2: relabel
      fused = m.relabel(points, offsets, poses, point_labels, keep_classes=things)
    m.save("map.npz")
"""
import os

import numpy as np
import torch

from . import _lib
from .device import ptr, require_cuda, stream_handle

HALF = 1 << 20     # voxel indices in [-2^20, 2^20)


def grown_capacity(capacity, fill, n):
  """The growth rule: before a vote of ``n`` points into a table of ``capacity`` slots holding ``fill`` keys, the
  capacity to vote into - unchanged while fill + n <= capacity / 2, else the smallest power of two >= 2 (fill + n).  The
  load then never passes 1/2 during a call."""
  need = int(fill) + int(n)
  if 2 * need <= capacity:
    return int(capacity)
  return 1 << (2 * need - 1).bit_length()


def unpack_keys(keys):
  """int64 / uint64 keys -> [V,3] int32 voxel indices."""
  k = np.asarray(keys).astype(np.int64)
  m = (1 << 21) - 1
  return np.stack([((k >> s) & m) - HALF for s in (42, 21, 0)], 1).astype(np.int32)


def kitti_lidar_poses(poses_txt, calib_txt):
  """SemanticKITTI poses in the lidar frame: [S,4,4] float64 ``inv(Tr) @ P_i @ Tr``, the composition semantic-kitti-api
  uses.  ``poses.txt`` holds one 3x4 camera pose per scan (12 numbers a line); ``Tr`` is the ``Tr:`` line of
  ``calib.txt`` (velodyne to camera)."""
  tr = None
  with open(calib_txt) as f:
    for line in f:
      key, _, vals = line.partition(":")
      if key.strip() == "Tr":
        tr = np.eye(4)
        tr[:3, :] = np.array(vals.split(), np.float64).reshape(3, 4)
  if tr is None:
    raise ValueError("%s has no Tr: line" % calib_txt)
  rows = np.loadtxt(poses_txt, dtype=np.float64, ndmin=2)
  if rows.shape[1] != 12:
    raise ValueError("%s: expected 12 numbers per line, got %d" % (poses_txt, rows.shape[1]))
  p = np.tile(np.eye(4), (rows.shape[0], 1, 1))
  p[:, :3, :] = rows.reshape(-1, 3, 4)
  out = np.linalg.inv(tr) @ p @ tr
  out[:, 3, :] = (0.0, 0.0, 0.0, 1.0)       # exact for rigid transforms; the inverse may leave rounding residue there
  return out


def scan_pose_index(path, num_poses):
  """The pose of a scan file is the integer stem of its name (``000123.bin`` -> 123), so that a glob over a subset of a
  sequence still finds its poses.  ValueError for a stem that is not a number or has no pose."""
  stem = os.path.splitext(os.path.basename(path))[0]
  if not stem.isdigit():
    raise ValueError("scan %s: the file stem is not a scan number, so it has no pose" % path)
  i = int(stem)
  if i >= num_poses:
    raise ValueError("scan %s: pose %d is out of range, the poses file has %d" % (path, i, num_poses))
  return i


class SemanticMap:
  """A voxel hash map of per-class vote counts on the GPU.

  num_classes   1..32; ``ignore_class`` (e.g. the "None" class) casts no vote, -1 = every class votes
  voxel_size    edge of a voxel in metres, in the world frame of the poses
  min_range, max_range  only points with min_range <= |p| (and |p| <= max_range when max_range > 0) in the sensor frame
                vote; queries are not limited
  capacity      initial slots, a power of two; the table grows by the rule of ``grown_capacity``

  The defaults (0.2 m voxels, 50 m, min_votes 1, thing classes kept by the CLI) are a starting point: they have not
  been tuned against real scans."""

  def __init__(self, num_classes, voxel_size=0.2, min_range=0.0, max_range=50.0, ignore_class=-1, capacity=1 << 20):
    self.num_classes, self.voxel_size = int(num_classes), float(voxel_size)
    self.min_range, self.max_range, self.ignore_class = float(min_range), float(max_range), int(ignore_class)
    capacity = int(capacity)
    if not 1 <= self.num_classes <= 32:
      raise ValueError("num_classes %d not in [1, 32]" % self.num_classes)
    if not (np.isfinite(self.voxel_size) and self.voxel_size > 0):
      raise ValueError("voxel_size %r must be finite and > 0" % voxel_size)
    if not (np.isfinite(self.min_range) and np.isfinite(self.max_range) and self.min_range >= 0
            and (self.max_range <= 0 or self.max_range >= self.min_range)):
      raise ValueError("range limits min %r max %r: need 0 <= min and max <= 0 (no limit) or max >= min"
                       % (min_range, max_range))
    if not (self.ignore_class == -1 or 0 <= self.ignore_class < self.num_classes):
      raise ValueError("ignore_class %d must be -1 or a class id" % self.ignore_class)
    if capacity < 1 or capacity & (capacity - 1):
      raise ValueError("capacity %d is not a power of two" % capacity)
    self._dev = require_cuda()
    self.state = torch.zeros(2, dtype=torch.int64, device=self._dev)
    self.keys, self.counts = self._table(capacity)

  @property
  def capacity(self):
    return int(self.keys.numel())

  def _table(self, capacity):
    keys = torch.full((capacity,), -1, dtype=torch.int64, device=self._dev)          # ~0 = empty
    return keys, torch.zeros((capacity, self.num_classes), dtype=torch.int32, device=self._dev)   # u32 counts

  def _state(self):
    """(occupied slots, failed inserts) - a device sync; raises if an insert found no free slot."""
    fill, failed = (int(v) for v in self.state.cpu())
    if failed:
      raise RuntimeError("semantic map: %d inserts found no free slot (the table overflowed)" % failed)
    return fill

  @property
  def num_voxels(self):
    return self._state()

  def _inputs(self, points, offsets, poses, labels):
    pts = _cuda(points, torch.float32)
    offs = _cuda(offsets, torch.int64)
    if pts.dim() != 2 or pts.shape[1] != 4:
      raise ValueError("points must be [total,4] float32 (x, y, z, remission)")
    B, total = int(offs.numel()) - 1, int(pts.shape[0])
    lab = _cuda(labels, torch.int32)
    if lab.numel() != total:
      raise ValueError("%d labels for %d points" % (lab.numel(), total))
    return pts, offs, _pose_rows(poses, B, self._dev), lab, B, total

  def vote(self, points, offsets, poses, labels):
    """Votes the labels of a batch of scans.  points [total,4] float32, offsets [B+1] int64, labels [total] int
    (numpy or CUDA), poses [B,4,4] float64 lidar-to-world (numpy or CUDA; finite, last row [0, 0, 0, 1])."""
    pts, offs, rows, lab, B, total = self._inputs(points, offsets, poses, labels)
    cap = grown_capacity(self.capacity, self._state(), total)
    if cap != self.capacity:
      self._grow(cap)
    lib = _lib.load()
    _lib.check(lib.pcls_semantic_map_vote(ptr(pts), ptr(offs), B, total, ptr(rows), self.voxel_size, self.min_range,
                                          self.max_range, ptr(lab), self.num_classes, self.ignore_class,
                                          ptr(self.keys), ptr(self.counts), self.capacity, ptr(self.state),
                                          stream_handle()), "pcls_semantic_map_vote")

  def _grow(self, capacity):
    keys, counts = self._table(capacity)
    _lib.check(_lib.load().pcls_semantic_map_grow(ptr(self.keys), ptr(self.counts), self.capacity, self.num_classes,
                                                  ptr(keys), ptr(counts), capacity, ptr(self.state), stream_handle()),
               "pcls_semantic_map_grow")
    self.keys, self.counts = keys, counts

  def relabel(self, points, offsets, poses, labels, keep_classes=(), min_votes=1):
    """[total] int32 CUDA: each point's label from the map - the argmax of its voxel's votes when the voxel has at
    least ``min_votes`` - except points whose label is one of ``keep_classes`` (e.g. the thing classes, which move and
    would be overwritten by the static votes under them) and points with no voxel in the map, which keep ``labels``."""
    pts, offs, rows, lab, B, total = self._inputs(points, offsets, poses, labels)
    self._state()
    if int(min_votes) < 1:
      raise ValueError("min_votes %r must be >= 1" % min_votes)
    mask = 0
    for c in keep_classes:
      if not 0 <= int(c) < self.num_classes:
        raise ValueError("keep class %r is not in [0, %d)" % (c, self.num_classes))
      mask |= 1 << int(c)
    out = torch.empty(total, dtype=torch.int32, device=self._dev)
    _lib.check(_lib.load().pcls_semantic_map_query(ptr(pts), ptr(offs), B, total, ptr(rows), self.voxel_size, ptr(lab),
                                                   self.num_classes, mask, int(min_votes), ptr(self.keys),
                                                   ptr(self.counts), self.capacity, ptr(out), stream_handle()),
               "pcls_semantic_map_query")
    return out

  def export(self):
    """dict(voxels [V,3] int32 voxel indices, counts [V,NC] uint32, labels [V] int32 = argmax of the counts with ties
    to the lowest class, voxel_size), sorted by key (x, then y, then z)."""
    self._state()
    occ = self.keys != -1
    keys = self.keys[occ]
    order = torch.argsort(keys)
    counts = self.counts[occ][order].cpu().numpy().view(np.uint32)
    keys = keys[order].cpu().numpy()
    labels = np.argmax(counts, axis=1).astype(np.int32) if len(keys) else np.zeros(0, np.int32)
    return dict(voxels=unpack_keys(keys), counts=counts, labels=labels, voxel_size=np.float64(self.voxel_size))

  def save(self, path):
    """Writes ``export()`` as an .npz file."""
    np.savez(path, **self.export())


def _cuda(x, dtype):
  t = x if torch.is_tensor(x) else torch.from_numpy(np.ascontiguousarray(x))
  return t.to(device=require_cuda(), dtype=dtype).contiguous()


def _pose_rows(poses, B, dev):
  """[B,4,4] float64 poses -> [B,12] float64 CUDA rows (R | t); ValueError unless finite with last row [0, 0, 0, 1]."""
  p = poses if torch.is_tensor(poses) else torch.from_numpy(np.asarray(poses))
  if p.dtype != torch.float64 or tuple(p.shape) != (B, 4, 4):
    raise ValueError("poses must be [%d,4,4] float64, got %s %s" % (B, tuple(p.shape), p.dtype))
  p = p.to(dev)
  last = torch.tensor([0.0, 0.0, 0.0, 1.0], dtype=torch.float64, device=dev)
  if not bool(torch.isfinite(p).all()) or not bool((p[:, 3, :] == last).all()):
    raise ValueError("poses must be finite rigid transforms with last row [0, 0, 0, 1]")
  return p[:, :3, :].reshape(B, 12).contiguous()
