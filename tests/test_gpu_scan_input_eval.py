"""The kernels on either side of the forward, per op, against bit-exact and float64 references:

  project_scatter_kernel                scan -> winner keys + per-point pixel (projection.cu), depth and ring variants
  project_resolve_kernel                keys -> [B,H,W,6] image, proj_idx, semantic label
  project_resolve_net_input_kernel<T>   keys -> the network's 16-bit input and mask byte, T = __half / __nv_bfloat16
  input_stage_kernel                    [n,5|6] sample -> normalised input, mask, int32 label, class weight
  cast_f64_f32_kernel, unpack_xyzir_kernel
  validation_kernel                     focal / sparse-CE loss sums and the weighted confusion matrix (validation.cu)
  confusion_kernel                      the confusion matrix of mIoU (confusion.cu)

Every kernel runs at least once past its grid cap (a grid-stride loop or a per-CTA chunk longer than one pass), computed
from the device's SM count; test_every_kernel_runs_past_its_cap checks that each one does, from the profiler's grids.

The projection cases plant points at pixel boundaries: for every column edge k in [0, W] and every row edge, float32
points within 4 * thr of the edge, where thr is the distance below which the kernel recomputes atan2 / asin in float64
(projection.cu).  Points inside thr are decided by the float64 path, points between thr and 4 thr by the float32 path
alone; both must give the correctly rounded pixel of oracle/projection.py (trig="cr").
"""
import ctypes
import os
import re
import time

import numpy as np
import pytest
import torch

from oracle import confusion as C
from oracle import nn as O
from oracle import projection as P
from pclsegmentation_b200 import _lib
from tests.util import synth_scan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32
PREC = {"f16": _lib.PCLS_F16, "bf16": _lib.PCLS_BF16}
KITTI = (64, 2048, 3.0, -25.0)
SENSORS = [KITTI, (64, 1024, 3.0, -25.0), (64, 512, 3.0, -25.0), (32, 1024, 12.0, -30.0)]   # nuScenes: 12 / -30
KITTI_MEAN, KITTI_STD = [-0.047, 0.365, -0.855, 0.2198, 8.3568], [10.154, 7.627, 0.8651, 0.1764, 9.6474]
NUSC_MEAN, NUSC_STD = [-0.1090, -0.1645, -0.6275, 17.2574, 11.5727], [11.4001, 12.9684, 1.9548, 20.2257, 12.9454]
BENCH_SCANS, BENCH_POINTS = 64, 120000        # bench.py projection_kitti_64x2048_b64: 64 scans of ~120 k points


def _s():
  return torch.cuda.current_stream().cuda_stream


def _sms():
  return torch.cuda.get_device_properties(0).multi_processor_count


def _d(a):
  return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _dbl(v):
  v = np.asarray(v, np.float64).reshape(-1)
  return (ctypes.c_double * v.size)(*v)


# ---- grid caps: elements one full grid covers in one pass (the launch code of each entry point) ---------------------
def cap_elems(kernel, sms):
  return {"project_scatter_kernel": sms * 16 * 256,       # grid_for: sm_count * 16 CTAs of 256; beyond: longer chunks
          "project_resolve_kernel": sms * 16 * 256,
          "project_resolve_net_input_kernel": sms * 16 * 256,
          "input_stage_kernel": sms * 16 * 256,
          "unpack_xyzir_kernel": sms * 16 * 256,
          "cast_f64_f32_kernel": sms * 16 * 256 * 2,       # a thread converts a pair
          "validation_kernel": sms * 6 * 8 * 32 * 4,       # sm_count * 6 CTAs, 8 warps of 32 px, 4 groups per warp
          "confusion_kernel": sms * 4 * 2048 * 4}[kernel]  # sm_count * 4 CTAs, 2048 int4 per CTA


def cap_grid(kernel, sms):
  return {"validation_kernel": sms * 6, "confusion_kernel": sms * 4}.get(kernel, sms * 16)


# ---- 16-bit rounding ------------------------------------------------------------------------------------------------
def to16(x, prec):
  """float32 -> the 16-bit pattern (uint16) of fp16 / bf16, round to nearest even; NaN -> a quiet NaN."""
  x = np.ascontiguousarray(x, dtype=F32)
  if prec == "f16":
    with np.errstate(over="ignore"):
      return x.astype(np.float16).view(np.uint16)
  b = x.view(np.uint32).astype(np.uint64)
  r = ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)
  return np.where(np.isnan(x), ((b >> 16) | 0x40).astype(np.uint16), r)


def _same16(a, b, prec):
  """uint16 patterns equal, or both NaN (a converted NaN's payload is not specified)."""
  a, b = np.asarray(a).view(np.uint16), np.asarray(b).view(np.uint16)
  nan = lambda v: (v & 0x7FFF) > (0x7C00 if prec == "f16" else 0x7F80)
  return (a == b) | (nan(a) & nan(b))


def test_to16_matches_torch():
  rng = np.random.default_rng(0)
  x = np.concatenate([rng.normal(0, 1e3, 20000), rng.normal(0, 1e-5, 5000), 2.0 ** rng.uniform(-140, 128, 5000)])
  x = x.astype(F32)
  ties = np.arange(1, 4000, dtype=np.uint32)
  x = np.concatenate([x, -x, (0x3F800000 + (ties << 12)).view(F32), (0x3F800000 + (ties << 15)).view(F32),
                      (0x3F800000 + (ties << 13) + 0x1000).view(F32), np.array([0.0, -0.0, np.inf, -np.inf, 65504,
                      65519.996, 65520, 6e-8, 2.9e-8, 3.0e-8, 3.4028235e38, 1e-45, np.nan], F32)]).astype(F32)
  for prec, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
    want = torch.from_numpy(x).to(dt).view(torch.int16).numpy().view(np.uint16)
    assert _same16(to16(x, prec), want, prec).all(), prec


# ---- A. projection: boundary points ---------------------------------------------------------------------------------
def proj_thr(H, W, fu, fd):
  """(thr_x, thr_y) of pcls_project_scatter, in float32 like the launch code."""
  fov = abs(fd / 180.0 * 3.141592653589793) + abs(fu / 180.0 * 3.141592653589793)
  thr_x = max(F32(1.5e-3), F32(7.5e-7) * F32(W))
  thr_y = max(F32(2e-4), F32(1.5e-6) * F32(H) / F32(fov) + F32(1.2e-6) * F32(H))
  return float(thr_x), float(thr_y)


def cr_fxy(pts, H, W, fu, fd):
  """Unclamped float32 column / row coordinates (fx, fy) of the correctly rounded projection (oracle, trig='cr')."""
  with np.errstate(all="ignore"):
    depth = P.point_depth(pts[:, :3])
    yaw, pitch = P.point_angles(pts[:, :3], depth, "cr")
    A, Fv = P._fov_constants(fu, fd)
    fx = F32(0.5) * (yaw / F32(np.pi) + F32(1.0)) * F32(W)
    fy = (F32(1.0) - (pitch + A) / Fv) * F32(H)
  return fx.astype(F32), fy.astype(F32)


def _edge_dist(f):
  with np.errstate(invalid="ignore"):
    return np.abs(f.astype(np.float64) - np.round(f.astype(np.float64)))


def _ulp_steps(a, steps):
  a = a.copy()
  for s in range(1, int(np.abs(steps).max(initial=0)) + 1):
    m = np.abs(steps) >= s
    a[m] = np.nextafter(a[m], np.where(steps[m] > 0, np.inf, -np.inf).astype(F32))
  return a


def _offsets(rng, n, thr):
  """Signed distances from an edge in pixels: half log-uniform in [1e-7, thr] (many within a float32 rounding of the
  edge), half uniform in [thr, 4 thr] (decided by the float32 path alone)."""
  inner = 10.0 ** rng.uniform(-7, np.log10(thr), n)
  outer = rng.uniform(thr, 4 * thr, n)
  return np.where(rng.random(n) < 0.5, inner, outer) * rng.choice([-1.0, 1.0], n)


def boundary_points(rng, H, W, fu, fd, per_col=12, per_row=None):
  """[n,4] float32 points whose correctly rounded fx (or fy) lies within 4 thr of a pixel edge, for every column edge
  k in [0, W] (0, W/2 and W included) and every row edge j in [0, H]; returns (points, is_column_point)."""
  thr_x, thr_y = proj_thr(H, W, fu, fd)
  A, Fv = (float(v) for v in P._fov_constants(fu, fd))
  lo, hi = np.deg2rad(fd) + 0.01, np.deg2rad(fu) - 0.01
  # columns: atan2(y, x) = -yaw = pi (1 - 2 (k + delta) / W)
  k = np.repeat(np.arange(W + 1), per_col)
  theta = np.pi * (1.0 - 2.0 * (k + _offsets(rng, k.size, thr_x)) / W)
  r, pitch = rng.uniform(1, 80, k.size), rng.uniform(lo, hi, k.size)
  col = np.stack([r * np.cos(pitch) * np.cos(theta), r * np.cos(pitch) * np.sin(theta), r * np.sin(pitch),
                  rng.random(k.size)], 1).astype(F32)
  for c in (0, 1):
    col[:, c] = _ulp_steps(col[:, c], rng.integers(-3, 4, k.size))
  # rows: pitch = (1 - (j + delta) / H) * fov - |fov_down|
  per_row = per_row or max(8, (W + 1) * per_col // (4 * (H + 1)))
  j = np.repeat(np.arange(H + 1), per_row)
  pitch = (1.0 - (j + _offsets(rng, j.size, thr_y)) / H) * Fv - A
  r, yaw = rng.uniform(1, 80, j.size), rng.uniform(-np.pi, np.pi, j.size)
  row = np.stack([r * np.cos(pitch) * np.cos(yaw), r * np.cos(pitch) * np.sin(yaw), r * np.sin(pitch),
                  rng.random(j.size)], 1).astype(F32)
  row[:, 2] = _ulp_steps(row[:, 2], rng.integers(-3, 4, j.size))
  fx, _ = cr_fxy(col, H, W, fu, fd)
  _, fy = cr_fxy(row, H, W, fu, fd)
  col, row = col[_edge_dist(fx) < 4 * thr_x], row[_edge_dist(fy) < 4 * thr_y]
  return np.concatenate([col, row]), np.arange(len(col) + len(row)) < len(col)


def special_points():
  """Signed zeros (x < 0 with y = +-0: yaw = -+pi, column 0 / W clamped to W-1), the origin, NaN / +-inf in each
  coordinate, pitch beyond the fov on both sides, tiny coordinates whose depth underflows to 0."""
  nan, inf = np.nan, np.inf
  p = [(0.0, 0.0, 1.0), (-0.0, 0.0, 1.0), (0.0, -0.0, 1.0), (-0.0, -0.0, 1.0), (-5.0, 0.0, 0.1), (-5.0, -0.0, 0.1),
       (-5.0, 0.0, -0.1), (-5.0, -0.0, -0.3), (5.0, 0.0, 0.0), (5.0, -0.0, -0.2), (0.0, 7.0, -1.0), (0.0, -7.0, -1.0),
       (-0.0, 7.0, 0.5), (0.0, 0.0, 0.0), (-0.0, -0.0, -0.0), (1e-30, 1e-30, 1e-30),
       (nan, 1.0, 1.0), (1.0, nan, 1.0), (1.0, 1.0, nan), (inf, 1.0, 0.0), (-inf, 1.0, 0.0), (1.0, inf, 0.0),
       (1.0, -inf, 0.0), (inf, inf, 0.0), (-inf, -inf, 0.0), (1.0, 1.0, inf), (1.0, 1.0, -inf), (inf, 0.0, inf),
       (10.0, 0.0, 50.0), (10.0, 0.0, -50.0), (0.0, 0.0, 5.0), (0.0, 0.0, -5.0), (3.0, 4.0, 0.9), (3.0, 4.0, -2.4),
       (1e30, 1e30, 1e30), (-2.0, 1e-38, 0.0)]
  pts = np.zeros((len(p), 4), F32)
  pts[:, :3] = np.array(p, F32)
  pts[:, 3] = np.linspace(0.05, 0.95, len(p))
  return pts


def test_boundary_generator_is_adversarial():
  """The projection cases need both bands: inside thr (the float64 path decides) and thr..4 thr (the float32 path
  alone decides), plus points on the float32 value next to an edge, where a 1-ulp error of atan2f / asinf moves the
  pixel; and every column edge, 0, W/2 and W included."""
  rng = np.random.default_rng(1)
  for H, W, fu, fd in SENSORS:
    pts, is_col = boundary_points(rng, H, W, fu, fd)
    thr_x, thr_y = proj_thr(H, W, fu, fd)
    fx, fy = cr_fxy(pts, H, W, fu, fd)
    for sel, f, thr in ((is_col, fx, thr_x), (~is_col, fy, thr_y)):
      d = _edge_dist(f[sel])
      assert (d < 4 * thr).all()
      assert (d < thr).mean() > 1 / 3 and ((d >= thr) & (d < 4 * thr)).mean() > 1 / 3, (H, W, (d < thr).mean())
      step = np.abs(np.spacing(np.round(f[sel]).astype(F32)))
      assert (d <= 2 * step).sum() > 0.02 * sel.sum(), (H, W, (d <= 2 * step).sum())
    edges = np.round(fx[is_col]).astype(np.int64)
    assert set(range(W + 1)) <= set(edges.tolist()), (H, W)
    rows = np.round(fy[~is_col]).astype(np.int64)
    assert set(range(H + 1)) <= set(rows.tolist()), (H, W)


# ---- A. projection: batches and expected values ---------------------------------------------------------------------
def _scan_sizes(rng, n_scans, mean_pts):
  """Ragged sizes: an empty first and last scan, a run of four empty scans, tiny scans with empty ones between them
  (one CTA chunk and one thread stride cross several scans), the rest around mean_pts."""
  sizes = rng.integers(int(mean_pts * 0.9), int(mean_pts * 1.1) + 1, n_scans)
  sizes[0] = sizes[-1] = 0
  sizes[5:9] = 0
  sizes[9:15] = [1, 0, 3, 0, 0, 5]
  return sizes


def make_batch(seed, H, W, fu, fd, n_scans, mean_pts, ring=False):
  """Synthetic scans with the boundary and special points planted, exact duplicates (depth ties) and, for the ring
  variant, ring values outside [0, H).  Returns (points [total,4] f32, ring [total] i32 or None, offsets [B+1] i64)."""
  rng = np.random.default_rng(seed)
  sizes = _scan_sizes(rng, n_scans, mean_pts)
  bpts, _ = boundary_points(rng, H, W, fu, fd)
  sp = special_points()
  big = np.flatnonzero(sizes > 100)
  share = np.array_split(rng.permutation(len(bpts)), len(big))
  scans, rings = [], []
  for b, n in enumerate(sizes):
    s = synth_scan(rng, int(n), fu, fd, H)
    if b in big:
      i = int(np.searchsorted(big, b))
      ins = bpts[share[i]]
      s = np.concatenate([s[: max(0, int(n) - len(ins))], ins])
      s = s[rng.permutation(len(s))]
      s[50:90] = s[0:40]                                    # exact duplicates: depth ties / ring collisions
      if i % 8 == 0:                                        # last: the zero-depth ones win their ring pixels
        s = np.concatenate([s, sp])
    scans.append(s)
    if ring:
      rg = rng.integers(0, H, len(s)).astype(np.int32)
      if len(s) > 100:
        rg[0:40] = rg[50:90] = rng.integers(0, H, 40)      # the duplicates collide in the same pixel
        rg[100:107] = [-1, H, H + 3, -7, 1 << 30, H - 1, 0]
      rings.append(rg)
  offsets = np.concatenate([[0], np.cumsum([len(s) for s in scans])]).astype(np.int64)
  return np.concatenate(scans).astype(F32), (np.concatenate(rings) if ring else None), offsets


def expected_projection(pts, ring, H, W, fu, fd):
  """Per-scan oracle of pcls_project_scatter's contract (pclseg.h): points with a non-finite pixel coordinate (or, in
  the ring variant, a row outside [0, H)) are dropped with proj_x = proj_y = -1; every other point and every pixel
  winner is P.range_projection / P.range_projection_ring (trig='cr') of the kept points.
  Returns (proj_x, proj_y, unproj_range, keys [H,W] u64, oracle dict with proj_idx in the scan's own indices)."""
  with np.errstate(all="ignore"):
    fx, fy = cr_fxy(pts, H, W, fu, fd)
    depth = P.point_depth(pts[:, :3])
  if ring is None:
    ok = np.isfinite(fx) & np.isfinite(fy)
  else:
    rows = (H - 1) - ring.astype(np.int64)
    ok = np.isfinite(fx) & (rows >= 0) & (rows < H)
  kept = np.flatnonzero(ok)
  with np.errstate(all="ignore"):
    if ring is None:
      o = P.range_projection(pts[kept, :3], pts[kept, 3], H, W, fu, fd, trig="cr")
    else:
      o = P.range_projection_ring(pts[kept, :3], pts[kept, 3], ring[kept], H, W, trig="cr")
  px = np.full(len(pts), -1, np.int32)
  py = np.full(len(pts), -1, np.int32)
  px[kept], py[kept] = o["proj_x"], o["proj_y"]
  occ = o["proj_idx"] >= 0
  idx = np.full((H, W), -1, np.int64)
  idx[occ] = kept[o["proj_idx"][occ]]
  o["proj_idx"] = idx.astype(np.int32)
  keys = np.full((H, W), np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64)
  lo = idx[occ].astype(np.uint64)
  hi = (o["proj_range"][occ].view(np.uint32).astype(np.uint64) if ring is None else (~lo) & np.uint64(0xFFFFFFFF))
  keys[occ] = (hi << np.uint64(32)) | lo
  return px, py, depth, keys, o


def _same_f32(a, b):
  a, b = np.asarray(a, F32), np.asarray(b, F32)
  return (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))


class Batch:
  """One scattered batch: device inputs, the kernel's outputs and the per-scan oracle."""

  def __init__(self, seed, sensor, n_scans, mean_pts, ring=False):
    self.H, self.W, self.fu, self.fd = sensor
    H, W = self.H, self.W
    self.pts, self.ring, self.off = make_batch(seed, H, W, self.fu, self.fd, n_scans, mean_pts, ring)
    self.B, self.total = len(self.off) - 1, int(self.off[-1])
    self.d_pts, self.d_off = _d(self.pts), _d(self.off)
    self.d_ring = _d(self.ring) if ring else None
    self.keys = torch.empty((self.B, H, W), dtype=torch.int64, device="cuda")
    self.px = torch.empty(self.total, dtype=torch.int32, device="cuda")
    self.py, self.ur = torch.empty_like(self.px), torch.empty(self.total, dtype=torch.float32, device="cuda")
    lib = _lib.load()
    _lib.check(lib.pcls_project_scatter(self.d_pts.data_ptr(), self.d_ring.data_ptr() if ring else None,
                                        self.d_off.data_ptr(), self.B, self.total, H, W, self.fu, self.fd,
                                        self.keys.data_ptr(), self.px.data_ptr(), self.py.data_ptr(),
                                        self.ur.data_ptr(), _s()), "pcls_project_scatter")
    torch.cuda.synchronize()
    self.ref = []
    for b in range(self.B):
      sl = slice(self.off[b], self.off[b + 1])
      self.ref.append(expected_projection(self.pts[sl], self.ring[sl] if ring else None, H, W, self.fu, self.fd))


_BATCHES = {}


def batch(name):
  """Module-wide cache: each batch is scattered and its oracle computed once."""
  if name not in _BATCHES:
    if name == "bench":
      _BATCHES[name] = Batch(11, KITTI, BENCH_SCANS, BENCH_POINTS * BENCH_SCANS // (BENCH_SCANS - 10))
    elif name == "ring":
      _BATCHES[name] = Batch(12, SENSORS[3], 24, 110000, ring=True)
    else:
      i = int(name[len("sensor"):])
      # 24 scans, 12 of them non-empty: about 1.5x the scatter's cap in all
      _BATCHES[name] = Batch(20 + i, SENSORS[i], 24, cap_elems("project_scatter_kernel", _sms()) // 8)
  return _BATCHES[name]


def _check_scatter(bt):
  keys = bt.keys.cpu().numpy().view(np.uint64)
  px, py, ur = bt.px.cpu().numpy(), bt.py.cpu().numpy(), bt.ur.cpu().numpy()
  for b in range(bt.B):
    sl = slice(bt.off[b], bt.off[b + 1])
    ex, ey, er, ek, _ = bt.ref[b]
    bad = np.flatnonzero(px[sl] != ex)
    assert bad.size == 0, "scan %d: proj_x differs at %d points, first %s: got %d, want %d" % (
        b, bad.size, bt.pts[sl][bad[0]], px[sl][bad[0]], ex[bad[0]])
    if bt.ring is None:
      bad = np.flatnonzero(py[sl] != ey)
      assert bad.size == 0, "scan %d: proj_y differs at %d points, first %s: got %d, want %d" % (
          b, bad.size, bt.pts[sl][bad[0]], py[sl][bad[0]], ey[bad[0]])
    else:
      assert np.array_equal(py[sl], np.where(ex >= 0, ey, -1))
    assert _same_f32(ur[sl], er).all(), "scan %d: unproj_range" % b
    bad = keys[b] != ek
    assert not bad.any(), "scan %d: keys differ at %d pixels" % (b, int(bad.sum()))


@pytest.mark.gpu
def test_projection_batch_layout_exercises_the_chunk_walk():
  """The bench-size batch runs capped (chunks longer than a CTA), one chunk holds the run of empty scans away from its
  start (the in-loop walk over several scans), and scans straddle chunk boundaries."""
  bt = batch("bench")
  sms = _sms()
  assert bt.total > cap_elems("project_scatter_kernel", sms)
  grid = min(-(-bt.total // 256), sms * 16)
  chunk = -(-bt.total // grid)
  assert chunk > 256
  off = bt.off
  run = off[5]
  assert (off[5:10] == run).all() and run % chunk != 0 and (off[15] // chunk) == (off[9] // chunk)
  assert sum(1 for b in range(bt.B) if off[b] // chunk != (off[b + 1] - 1) // chunk and off[b + 1] > off[b]) > 30


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bench", "sensor1", "sensor2", "sensor3"])
def test_project_scatter_bit_exact_at_pixel_boundaries(name):
  """Depth variant: proj_x, proj_y, unproj_range and the winner keys (min depth, then lowest index) bit-equal to the
  correctly rounded oracle on boundary, special and duplicate points, for each sensor; 'bench' is the benchmark's
  projection workload (64 scans, KITTI 64x2048)."""
  bt = batch(name)
  assert bt.total > cap_elems("project_scatter_kernel", _sms())
  _check_scatter(bt)
  # the special points were dropped / clamped as the contract says
  sp = special_points()
  ex, ey, _, _, _ = expected_projection(sp, None, bt.H, bt.W, bt.fu, bt.fd)
  assert (ex[13:15] == -1).all() and (ex[16:19] == -1).all() and ex[19] == bt.W // 2 and ex[20] == 0
  assert ex[4] == 0 and ex[5] == bt.W - 1 and ey[28] == 0 and ey[29] == bt.H - 1 and ex[27] == -1


@pytest.mark.gpu
def test_project_scatter_ring_variant():
  """Ring variant vs P.range_projection_ring: rows from the ring index, ring values outside [0, H) dropped with -1,
  zero-depth points kept (the origin wins its pixel), collisions won by the highest index."""
  bt = batch("ring")
  assert bt.total > cap_elems("project_scatter_kernel", _sms())
  _check_scatter(bt)
  keys = bt.keys.cpu().numpy().view(np.uint64)
  px = bt.px.cpu().numpy()
  ring_bad = (bt.ring < 0) | (bt.ring >= bt.H)
  assert ring_bad.sum() >= 5 * 10 and (px[ring_bad] == -1).all()
  zero = np.flatnonzero((bt.ur.cpu().numpy() == 0) & (px >= 0))
  assert zero.size > 0, "no zero-depth point was kept"
  b_of = np.searchsorted(bt.off, zero, side="right") - 1
  win = [(keys[b, (bt.H - 1) - bt.ring[z], px[z]] & 0xFFFFFFFF) for b, z in zip(b_of, zero)]
  assert any(int(w) == z - bt.off[b] for w, z, b in zip(win, zero, b_of)), "no zero-depth point won its pixel"
  coll = 0
  for b in range(bt.B):
    if bt.off[b + 1] - bt.off[b] > 100:                    # the duplicates 0..39 / 50..89 share their pixels
      sl = slice(bt.off[b], bt.off[b + 1])
      p0 = px[sl][:40]
      r0 = (bt.H - 1) - bt.ring[sl][:40]
      ok = (p0 >= 0) & (r0 >= 0) & (r0 < bt.H)
      w = keys[b][r0[ok], p0[ok]] & np.uint64(0xFFFFFFFF)
      coll += int((w >= 50).sum())
      assert (w >= 50).all()
  assert coll > 100


# ---- B. scan -> network input ---------------------------------------------------------------------------------------
def _mean_std(bt):
  return (NUSC_MEAN, NUSC_STD) if bt.ring is not None or bt.H == 32 else (KITTI_MEAN, KITTI_STD)


def expected_net_input(bt, b, prec):
  """P.assemble_range_image (empty fill 0) -> O.input_stage -> 16-bit round to nearest even; channel 5 = mask,
  channels 6, 7 = 0.  Returns (uint16 [H,W,8], mask u8 [H,W], proj_idx [H,W])."""
  o = bt.ref[b][4]
  mean, std = _mean_std(bt)
  with np.errstate(all="ignore"):
    img = P.assemble_range_image(o).astype(F32)
    lidar, mask, _ = O.input_stage(img, mean, std, 0)
  h = np.zeros((bt.H, bt.W, 8), np.uint16)
  h[..., :6] = to16(lidar, prec)
  return h, mask.astype(np.uint8), o["proj_idx"]


def run_net_input(bt, b0, b1, prec, with_idx=True):
  lib = _lib.load()
  B, H, W = b1 - b0, bt.H, bt.W
  mean, std = _mean_std(bt)
  inp = torch.full((B, H, W, 8), -1, dtype=torch.int16, device="cuda")
  msk = torch.full((B, H, W), 7, dtype=torch.uint8, device="cuda")
  idx = torch.full((B, H, W), -5, dtype=torch.int32, device="cuda") if with_idx else None
  _lib.check(lib.pcls_project_resolve_net_input(bt.d_pts.data_ptr(), bt.d_off[b0:].data_ptr(), B, H, W,
                                                bt.keys[b0:].data_ptr(), _dbl(mean), _dbl(std), PREC[prec],
                                                inp.data_ptr(), msk.data_ptr(), idx.data_ptr() if with_idx else None,
                                                _s()), "pcls_project_resolve_net_input")
  torch.cuda.synchronize()
  return (inp.cpu().numpy().view(np.uint16), msk.cpu().numpy(), idx.cpu().numpy() if with_idx else None)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", list(PREC))
@pytest.mark.parametrize("case", ["bench32", "one", "empty", "ring"])
def test_project_resolve_net_input_bit_exact(case, prec):
  """The fused keys -> 16-bit network input: [B,H,W,8] pixels, mask byte and proj_idx bit-equal to the oracle chain;
  32x64x2048 runs past the grid cap, 'one' and 'empty' are 1xHxW (a scan with points, the empty first scan), 'ring'
  has zero-depth winners (mask 0, inputs 0, proj_idx set) and NaN-depth winners; the special points put +-inf
  coordinates in the bench batch.  proj_idx = NULL writes the same input and mask."""
  bt = batch("ring" if case == "ring" else "bench")
  b0, b1 = {"bench32": (0, 32), "one": (15, 16), "empty": (0, 1), "ring": (0, bt.B)}[case]
  if case == "bench32":
    assert (b1 - b0) * bt.H * bt.W > cap_elems("project_resolve_net_input_kernel", _sms())
  inp, msk, idx = run_net_input(bt, b0, b1, prec)
  inp2, msk2, _ = run_net_input(bt, b0, b1, prec, with_idx=False)
  assert np.array_equal(inp, inp2) and np.array_equal(msk, msk2)
  n_inf = n_zero = 0
  for b in range(b0, b1):
    h, m, i = expected_net_input(bt, b, prec)
    bad = ~_same16(inp[b - b0], h, prec)
    assert not bad.any(), "scan %d: input differs at %d elements, first %s" % (b, int(bad.sum()), np.argwhere(bad)[0])
    assert np.array_equal(msk[b - b0], m) and np.array_equal(idx[b - b0], i)
    n_inf += int(((inp[b - b0][..., :5] & 0x7FFF) == (0x7C00 if prec == "f16" else 0x7F80)).sum())
    n_zero += int(((i >= 0) & (m == 0)).sum())
  if case == "bench32":
    assert n_inf > 0, "no +-inf coordinate reached the network input"
  if case == "ring":
    assert n_zero > 0, "no zero-depth winner"
  if case == "empty":
    assert (idx == -1).all() and (msk == 0).all() and (inp == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("prec", list(PREC))
@pytest.mark.parametrize("name", ["bench", "ring"])
def test_fused_net_input_equals_staged_path(name, prec):
  """On the same keys, pcls_project_resolve_net_input writes the bytes the staged path writes:
  pcls_project_resolve (empty fill 0) -> pcls_input_stage -> the net's input kernel, read back raw through
  pcls_net_input_buffers.  Per pixel, not only the logits downstream."""
  from tests import test_gpu_cam_pool_input as CP
  bt = batch(name)
  b0, b1 = (15, 17) if name == "bench" else (1, 3)
  B, H, W = b1 - b0, bt.H, bt.W
  lib = _lib.load()
  mean, std = _mean_std(bt)
  img = torch.empty((B, H, W, 6), dtype=torch.float32, device="cuda")
  _lib.check(lib.pcls_project_resolve(bt.d_pts.data_ptr(), None, bt.d_off[b0:].data_ptr(), B, H, W,
                                      bt.keys[b0:].data_ptr(), None, 0, 0.0, img.data_ptr(), None, None, _s()),
             "pcls_project_resolve")
  lidar = torch.empty((B, H, W, 6), dtype=torch.float32, device="cuda")
  _lib.check(lib.pcls_input_stage(img.data_ptr(), 6, B * H * W, _dbl(mean), _dbl(std), 0, lidar.data_ptr(), None,
                                  None, None, 0, None, _s()), "pcls_input_stage")
  net = CP._InputNet(prec, B, H, W)
  try:
    t0, m, _ = net.run(lidar.cpu(), 6)
  finally:
    net.close()
  inp, msk, _ = run_net_input(bt, b0, b1, prec)
  staged = t0.cpu().numpy().view(np.uint16)
  bad = ~_same16(staged, inp, prec)
  assert not bad.any(), "fused and staged inputs differ at %d elements" % int(bad.sum())
  assert np.array_equal(m.cpu().numpy(), msk)


@pytest.mark.gpu
def test_project_resolve_labels_lut_and_empty_fill():
  """pcls_project_resolve: LUT ids >= lut_len map to 0, the upper 16 label bits are ignored, labels = NULL gives
  sem 0 (LUT[0] in the image), and a zero-depth winner keeps its values with empty_fill -1 but is zeroed with 0."""
  bt = batch("ring")
  lib = _lib.load()
  B, H, W = bt.B, bt.H, bt.W
  rng = np.random.default_rng(3)
  sem = rng.integers(0, 40, bt.total).astype(np.uint32)
  labels = sem | (rng.integers(1, 1 << 16, bt.total).astype(np.uint32) << 16)
  lut_len = 25
  lut = (np.arange(lut_len, dtype=np.int32) * 7 + 3)
  d_lab, d_lut = _d(labels.view(np.int32)), _d(lut)
  zero_winners = 0
  for fill in (-1.0, 0.0):
    for use_labels in (True, False):
      img = torch.empty((B, H, W, 6), dtype=torch.float32, device="cuda")
      idx = torch.empty((B, H, W), dtype=torch.int32, device="cuda")
      ps = torch.empty((B, H, W), dtype=torch.int32, device="cuda")
      _lib.check(lib.pcls_project_resolve(bt.d_pts.data_ptr(), d_lab.data_ptr() if use_labels else None,
                                          bt.d_off.data_ptr(), B, H, W, bt.keys.data_ptr(), d_lut.data_ptr(), lut_len,
                                          fill, img.data_ptr(), idx.data_ptr(), ps.data_ptr(), _s()),
                 "pcls_project_resolve")
      img, idx, ps = img.cpu().numpy(), idx.cpu().numpy(), ps.cpu().numpy()
      for b in range(B):
        o = bt.ref[b][4]
        sl = slice(bt.off[b], bt.off[b + 1])
        s = P.label_projection(o["proj_idx"], labels[sl]) if use_labels else np.zeros((H, W), np.int32)
        assert np.array_equal(idx[b], o["proj_idx"]) and np.array_equal(ps[b], s)
        mapped = np.where(s < lut_len, lut[np.minimum(s, lut_len - 1)], 0).astype(F32)
        if fill == 0.0:
          with np.errstate(invalid="ignore"):
            ref = P.assemble_range_image(o).astype(F32)
        else:
          ref = np.concatenate([o["proj_xyz"], o["proj_remission"][..., None], o["proj_range"][..., None],
                                np.zeros((H, W, 1))], -1).astype(F32)
        ref[..., 5] = mapped
        assert _same_f32(img[b], ref).all(), "scan %d fill %g labels %s" % (b, fill, use_labels)
        zw = (o["proj_idx"] >= 0) & ~(o["proj_range"] > 0)
        zero_winners += int(zw.sum())
        if fill == -1.0 and zw.any():
          assert (img[b][zw][:, 3] != 0).any()             # the remission of a zero-depth winner survives with -1
  assert zero_winners > 0
  assert (sem >= lut_len).mean() > 0.3


# ---- C. input stage --------------------------------------------------------------------------------------------------
EDGE_RANGE = np.array([-0.0, np.nan, 1e-40, -1e-40, 0.0, 2.0], F32)
EDGE_LABEL = np.array([2.5, -1.0, -0.5, 20.0, 31.0, 1e10, -1e10, np.nan, -0.0, np.inf, 3.0, 19.0, 19.999, 0.0], F32)


def input_stage_sizes(sms):
  cap = cap_elems("input_stage_kernel", sms)
  return [1, cap - 1, cap, cap + 1, 32 * 64 * 2048]


def _input_sample(rng, n, channels, nc):
  x = np.empty((n, channels), F32)
  x[:, :4] = rng.normal(0, 20, (n, 4))
  x[:, 4] = np.where(rng.random(n) < 0.75, rng.uniform(1, 80, n), 0.0)
  if channels == 6:
    x[:, 5] = rng.integers(0, nc, n)
  # edge values at valid and masked pixels
  k = min(n, 4000)
  i = rng.permutation(n)[:k]
  x[i[: k // 2], 4] = rng.choice(EDGE_RANGE, k // 2)
  if channels == 6:
    x[i[k // 4:], 5] = rng.choice(EDGE_LABEL, k - k // 4)
  x[0, 4] = 1e-40
  if channels == 6:
    x[0, 5] = 2.5                                          # pixel 0: valid (subnormal range) with a fractional label
  return x


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [5, 6])
@pytest.mark.parametrize("size", range(5), ids=["1", "cap-1", "cap", "cap+1", "32x64x2048"])
def test_input_stage_bit_exact(size, channels):
  """pcls_input_stage vs O.input_stage and the label rule of pclseg.h, with -0.0 / NaN / subnormal ranges and
  fractional, negative, >= NC, NaN, +-inf and -0.0 labels at valid and masked pixels, distinct class weights, and each
  output NULL in turn (the others must not change)."""
  n = input_stage_sizes(_sms())[size]
  nc, none = 20, 19
  rng = np.random.default_rng(n + channels)
  x = _input_sample(rng, n, channels, nc)
  cls_w = np.linspace(0.25, 3.0, nc)
  lib = _lib.load()
  d = _d(x)
  x6 = x if channels == 6 else np.concatenate([x, np.zeros((n, 1), F32)], 1)
  with np.errstate(invalid="ignore"):
    lid_ref, m_ref, lab_ref = O.input_stage(x6.reshape(n, 1, 6), KITTI_MEAN, KITTI_STD, none)
    w_ref = O.class_weight_map(O.fixed_label(x6.reshape(n, 1, 6), none), cls_w).reshape(n)
  lid_ref, m_ref, lab_ref = lid_ref.reshape(n, 6), m_ref.reshape(n).astype(np.uint8), lab_ref.reshape(n)
  outs = ("lidar", "mask", "label", "weight") if channels == 6 else ("lidar", "mask")
  for null in (None,) + outs:
    t = {"lidar": torch.full((n, 6), 7.0, device="cuda"), "mask": torch.full((n,), 9, dtype=torch.uint8, device="cuda"),
         "label": torch.full((n,), -9, dtype=torch.int32, device="cuda"),
         "weight": torch.full((n,), 7.0, device="cuda")}
    ptr = {k: (None if (k == null or k not in outs) else v.data_ptr()) for k, v in t.items()}
    _lib.check(lib.pcls_input_stage(d.data_ptr(), channels, n, _dbl(KITTI_MEAN), _dbl(KITTI_STD), none, ptr["lidar"],
                                    ptr["mask"], ptr["label"], _dbl(cls_w) if ptr["weight"] else None, nc,
                                    ptr["weight"], _s()), "pcls_input_stage")
    got = {k: v.cpu().numpy() for k, v in t.items()}
    for k, ref in (("lidar", lid_ref), ("mask", m_ref), ("label", lab_ref), ("weight", w_ref)):
      if ptr[k] is None:
        assert (got[k] == t[k][:1].cpu().numpy()[0]).all(), "%s written although NULL" % k
        continue
      if k in ("lidar", "weight"):
        bad = ~_same_f32(got[k], ref)
      else:
        bad = got[k] != ref
      assert not bad.any(), "%s differs at %d elements, first at %s" % (k, int(bad.sum()), np.argwhere(bad)[0])
  if channels == 6 and n > 1000:
    valid = m_ref.astype(bool)
    lf = x[:, 5]
    assert ((lf == 2.5) & valid).any() and ((np.isnan(lf)) & valid).any() and ((lf >= nc) & valid).any()
    assert w_ref[0] == 0 and lab_ref[0] == 2                # 2.5: label 2, weight 0 (the float is no class)


def test_label_rule_of_the_oracle():
  """O.label_to_int32 / O.class_weight_map state pclseg.h's rule without the GPU."""
  lf = np.array([2.5, -0.5, -1.0, np.nan, -0.0, 1e10, -1e10, np.inf, 3.0, 19.999], F32)
  assert O.label_to_int32(lf).tolist() == [2, 0, -1, 0, 0, 2 ** 31 - 1, -2 ** 31, 2 ** 31 - 1, 3, 19]
  w = O.class_weight_map(lf, np.arange(1, 21, dtype=np.float64))
  assert w.tolist() == [0, 0, 0, 0, 1, 0, 0, 0, 4, 0]


# ---- D. validation and confusion -------------------------------------------------------------------------------------
def _probs(n, nc, seed):
  g = torch.Generator(device="cuda").manual_seed(seed)
  logits = torch.randn((n, nc), generator=g, device="cuda") * 3
  p = torch.softmax(logits, 1)
  p[: n // 50] = torch.softmax(logits[: n // 50] * 8, 1)   # near-one-hot rows: p close to 1, (1 - p) tiny
  return p.contiguous()


def _sce_row_sums(p32):
  """sum_c clip(p_c) in float32, classes in order: the kernel's own sum, so that only the logs differ."""
  c = np.clip(p32, F32(1e-7), F32(1.0 - 1e-7))
  s = np.zeros(len(c), F32)
  for j in range(c.shape[1]):
    s = s + c[:, j]
  return s, c


def validation_refs(probs, label, pred, mask, weight, nc, eps, gamma, chunk=1 << 20):
  """float64 sums of the per-pixel terms computed from the kernel's float32 values.  Focal: p = f32(probs[y] + eps),
  a = f32(1 - p), term = a^gamma * -log(p); sparse CE: s = the float32 class sum, term = log(s) - log(clip(p[y])).
  Returns dict: kind -> (num, sum of |term| w m, sum of (|log s| + |log py|) w), per (use_mask, use_w)."""
  n = len(label)
  acc = {}
  for a in range(0, n, chunk):
    sl = slice(a, min(n, a + chunk))
    p = probs[sl]
    y = label[sl]
    ok = (y >= 0) & (y < nc)
    yc = np.where(ok, y, 0)
    py = p[np.arange(len(y)), yc]
    pe = (py + F32(eps)).astype(F32)
    one_m = (F32(1.0) - pe).astype(F32)
    with np.errstate(divide="ignore"):
      focal = np.where(ok, one_m.astype(np.float64) ** gamma * -np.log(pe.astype(np.float64)), 0.0)
    s, cl = _sce_row_sums(p)
    pyc = cl[np.arange(len(y)), yc]
    ls, lp = np.log(s.astype(np.float64)), np.log(pyc.astype(np.float64))
    sce = np.where(ok, ls - lp, 0.0)
    sce_mag = np.where(ok, np.abs(ls) + np.abs(lp), 0.0)
    for um in (True, False):
      for uw in (True, False):
        m = mask[sl].astype(np.float64) if um else 1.0
        w = weight[sl].astype(np.float64) if uw else 1.0
        key = (um, uw)
        r = acc.setdefault(key, np.zeros(6))
        r += [(focal * w * m).sum(), (np.abs(focal) * w * m).sum(), (sce * w).sum(), (np.abs(sce) * w).sum(),
              (sce_mag * w).sum(), np.sum(m * np.ones(len(y)))]
  return acc


def _validation_case_sizes(sms):
  cap = cap_elems("validation_kernel", sms)
  return {"eval-20": (32 * 64 * 2048, 20), "4cap-20": (4 * cap + 17, 20), "4cap-32": (4 * cap + 29, 32)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["eval-20", "4cap-20", "4cap-32", "labels-out", "all-masked"])
def test_validation_update_past_the_cap(case):
  """pcls_validation_update at the eval step's shape (32x64x2048, NC 20) and ~4x the grid cap (NC 20, 32), both loss
  kinds, the mask and the weights each absent, out-of-range labels / predictions; every label out of range and every
  pixel masked out (den = 0); eps = the shipped DENOM_EPSILON.

  Tolerance of the loss sums (all terms are >= 0 for focal, the sparse-CE logs are bounded term by term):
    focal: the kernel's term is powf(a, gamma) * -logf(p) in float32: powf <= 4 ulp, logf <= 1 ulp, the product 0.5 ulp
           (CUDA C Programming Guide, maximum ulp errors), so |dterm| <= 5.5 * 2^-23 * term (+ a rounding of the 2^-24
           order per factor, inside the margin); float64 accumulation in any order adds <= n * 2^-53 of the sum of |terms|.
    sparse CE: logf(s) and logf(p_y) each <= 1 ulp <= 2^-23 |log|, the class sum s is the kernel's own float32 sum, so
           |dterm| <= 2^-23 (|log s| + |log p_y|) w, plus the float64 accumulation as above.
  The weighted confusion matrix is a float64 sum of float32 weights: 1e-12 relative; dropped exactly."""
  from pclsegmentation_b200.configs import SqueezeSegV2KittiConfig
  mc = SqueezeSegV2KittiConfig()
  eps, gamma = float(mc.DENOM_EPSILON), float(mc.FOCAL_GAMMA)
  sms = _sms()
  sizes = _validation_case_sizes(sms)
  n, nc = sizes.get(case, (2 * cap_elems("validation_kernel", sms) + 3, 20))
  assert n > cap_elems("validation_kernel", sms)
  rng = np.random.default_rng(n + nc)
  P_ = _probs(n, nc, n)
  probs = P_.cpu().numpy()
  label = rng.integers(0, nc, n).astype(np.int32)
  pred = np.where(rng.random(n) < 0.7, label, rng.integers(0, nc, n)).astype(np.int32)
  bad = rng.random(n) < 0.01
  label[bad] = rng.choice(np.array([-1, nc, nc + 5, -(1 << 30)], np.int32), int(bad.sum()))
  pred[rng.random(n) < 0.01] = nc
  mask = (rng.random(n) < 0.7).astype(np.uint8)
  if case == "labels-out":
    label[:] = np.where(rng.random(n) < 0.5, nc, -1)
  if case == "all-masked":
    mask[:] = 0
  weight = rng.uniform(0.2, 3.0, n).astype(F32)
  Y, Q, M, Wt = _d(label), _d(pred), _d(mask), _d(weight)
  lib = _lib.load()

  def run(kind, um, uw, cm_on):
    acc = torch.zeros(2, dtype=torch.float64, device="cuda")
    cm = torch.zeros((nc, nc), dtype=torch.float64, device="cuda") if cm_on else None
    dr = torch.zeros(1, dtype=torch.int64, device="cuda")
    _lib.check(lib.pcls_validation_update(P_.data_ptr(), Y.data_ptr(), Q.data_ptr() if cm_on else None,
                                          M.data_ptr() if um else None, Wt.data_ptr() if uw else None, n, nc, kind,
                                          eps, gamma, acc.data_ptr(), cm.data_ptr() if cm_on else None,
                                          dr.data_ptr() if cm_on else None, _s()), "pcls_validation_update")
    return acc.cpu().numpy(), (cm.cpu().numpy() if cm_on else None), int(dr.item())

  refs = validation_refs(probs, label, pred, mask, weight, nc, eps, gamma)
  okp = (label >= 0) & (label < nc) & (pred >= 0) & (pred < nc)
  for um, uw in ((True, True), (False, True), (True, False), (False, False)):
    focal, focal_abs, sce, sce_abs, sce_mag, den = refs[(um, uw)]
    acc, cm, dr = run(1, um, uw, True)
    tol = 5.5 * 2.0 ** -23 * focal_abs + n * 2.0 ** -53 * focal_abs
    assert abs(acc[0] - focal) <= tol, ("focal", um, uw, acc[0], focal, tol)
    assert acc[1] == den, ("focal den", um, uw, acc[1], den)
    w = weight.astype(np.float64) if uw else np.ones(n)
    ref = np.bincount(label[okp].astype(np.int64) * nc + pred[okp], weights=w[okp], minlength=nc * nc).reshape(nc, nc)
    assert np.allclose(cm, ref, rtol=1e-12, atol=0) and dr == int((~okp).sum())
    if um:
      continue
    acc, cm2, _ = run(2, False, uw, not uw)
    tol = 2.0 ** -23 * sce_mag + n * 2.0 ** -53 * sce_abs
    assert abs(acc[0] - sce) <= tol, ("sce", uw, acc[0], sce, tol)
    assert acc[1] == n
  if case == "all-masked":
    assert refs[(True, True)][5] == 0
  if case == "labels-out":
    assert refs[(True, True)][0] == 0 and refs[(False, True)][2] == 0


def confusion_cases(sms):
  cap = cap_elems("confusion_kernel", sms)
  big = 64 * 64 * 2048
  return {"64x64x2048-20": (big, 20, "skew"), "64x64x2048-32": (big, 32, "skew"), "cap2+1": (2 * cap + 1, 20, "skew"),
          "cap2+2": (2 * cap + 2, 20, "skew"), "cap2+3": (2 * cap + 3, 32, "skew"), "flood": (big + 3, 20, "flood")}


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["64x64x2048-20", "64x64x2048-32", "cap2+1", "cap2+2", "cap2+3", "flood"])
def test_confusion_update_past_the_cap(case):
  """pcls_confusion_update bit-exact vs C.confusion_matrix past its grid cap (Darknet53's eval batch of 64 frames),
  NC 20 and 32, the scalar tail of n % 4 = 1, 2, 3 past the cap, out-of-range pairs counted, and a flood where every
  pixel is the same bin (a whole warp per __match_any_sync group).  Accumulates across two calls like update_state."""
  n, nc, kind = confusion_cases(_sms())[case]
  assert n > cap_elems("confusion_kernel", _sms())
  rng = np.random.default_rng(n + nc)
  if kind == "flood":
    label = np.full(n, nc - 1, np.int32)
    pred = np.full(n, nc - 1, np.int32)
  else:
    p = np.full(nc, 0.5 / (nc - 1))
    p[nc - 1] = 0.5
    label = rng.choice(nc, n, p=p / p.sum()).astype(np.int32)
    pred = np.where(rng.random(n) < 0.8, label, rng.integers(0, nc, n)).astype(np.int32)
    bad = rng.random(n) < 1e-3
    label[bad] = rng.choice(np.array([-1, nc, 1 << 20], np.int32), int(bad.sum()))
  t = n - n % 4
  label[t:] = np.arange(n - t) % nc                         # the tail: valid, distinct bins
  pred[t:] = (np.arange(n - t) * 3 + 1) % nc
  lib = _lib.load()
  L, Pd = _d(label), _d(pred)
  cm = torch.zeros((nc, nc), dtype=torch.int64, device="cuda")
  dr = torch.zeros(1, dtype=torch.int64, device="cuda")
  for _ in range(2):
    _lib.check(lib.pcls_confusion_update(L.data_ptr(), Pd.data_ptr(), n, nc, cm.data_ptr(), dr.data_ptr(), _s()),
               "pcls_confusion_update")
  ok = (label >= 0) & (label < nc) & (pred >= 0) & (pred < nc)
  ref = C.confusion_matrix(label[ok], pred[ok], nc)
  got = cm.cpu().numpy()
  assert np.array_equal(got, 2 * ref), "cm differs in %d bins" % int((got != 2 * ref).sum())
  assert int(dr.item()) == 2 * int((~ok).sum())


# ---- E. small kernels ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cast_f64_f32_past_the_cap():
  """pcls_cast_f64_f32 bit-equal to numpy astype past its grid cap, odd length, specials at both ends."""
  sms = _sms()
  n = 2 * cap_elems("cast_f64_f32_kernel", sms) + 3
  rng = np.random.default_rng(7)
  x = rng.normal(0, 50, n) * 10.0 ** rng.integers(-40, 40, n)
  sp = [0.1, -1e-45, 3.4028235677973366e38, 1e39, -np.inf, 16777217.0, 1.0000000596046448, -0.0, 1e-46, np.nan]
  x[:len(sp)] = sp
  x[-len(sp):] = sp[::-1]
  out = torch.empty(n, dtype=torch.float32, device="cuda")
  d = _d(x)
  _lib.check(_lib.load().pcls_cast_f64_f32(d.data_ptr(), out.data_ptr(), n, _s()), "pcls_cast_f64_f32")
  with np.errstate(over="ignore"):
    want = x.astype(F32)
  assert _same_f32(out.cpu().numpy(), want).all()


@pytest.mark.gpu
@pytest.mark.parametrize("with_ring", [True, False])
def test_unpack_xyzir_past_the_cap(with_ring):
  """pcls_unpack_xyzir vs numpy: the [n,4] points and ring = astype(np.int32), truncation toward zero (31.9 -> 31,
  -0.5 -> 0, 63.0 -> 63), odd n past the cap, ring = NULL."""
  sms = _sms()
  n = 2 * cap_elems("unpack_xyzir_kernel", sms) + 1
  rng = np.random.default_rng(8)
  rec = rng.normal(0, 30, (n, 5)).astype(F32)
  rec[:, 4] = rng.uniform(-0.99, 64, n)
  rec[:8, 4] = [31.9, -0.5, 63.0, 0.0, -0.0, 0.999, 31.0, 32.5]
  rec[-3:, 4] = [63.99, -0.999, 12.0]
  pts = torch.full((n, 4), 5.0, device="cuda")
  ring = torch.full((n,), -9, dtype=torch.int32, device="cuda")
  d = _d(rec)
  _lib.check(_lib.load().pcls_unpack_xyzir(d.data_ptr(), n, pts.data_ptr(), ring.data_ptr() if with_ring else None,
                                           _s()), "pcls_unpack_xyzir")
  assert np.array_equal(pts.cpu().numpy().view(np.uint32), rec[:, :4].copy().view(np.uint32))
  r = ring.cpu().numpy()
  if with_ring:
    assert np.array_equal(r, rec[:, 4].astype(np.int32)) and r[:3].tolist() == [31, 0, 63]
  else:
    assert (r == -9).all()


# ---- F. coverage guard -----------------------------------------------------------------------------------------------
CSRC = os.path.join(ROOT, "pclsegmentation_b200", "csrc")
GUARDED = ("projection.cu", "input_stage.cu", "validation.cu", "confusion.cu")


def source_kernels():
  """{(kernel, template argument or None)} launched in the guarded sources."""
  out = set()
  for f in GUARDED:
    with open(os.path.join(CSRC, f)) as fh:
      src = fh.read()
    defined = set(re.findall(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s*)?(\w+)\s*\(", src))
    launched = {(name, targ or None) for name, targ in re.findall(r"(\w+_kernel)(?:<([\w:]+)>)?<<<", src)}
    assert defined and defined == {k for k, _ in launched}, (f, defined, launched)
    out |= launched
  return out


# every kernel, with every instantiation, and the tests above that launch it past its cap
CASES = {("project_scatter_kernel", None): "test_project_scatter_bit_exact_at_pixel_boundaries[bench], ring variant",
         ("project_resolve_kernel", None): "test_project_resolve_labels_lut_and_empty_fill",
         ("project_resolve_net_input_kernel", "__half"): "test_project_resolve_net_input_bit_exact[bench32-f16]",
         ("project_resolve_net_input_kernel", "__nv_bfloat16"): "test_project_resolve_net_input_bit_exact[bench32-bf16]",
         ("input_stage_kernel", None): "test_input_stage_bit_exact[cap+1 / 32x64x2048]",
         ("cast_f64_f32_kernel", None): "test_cast_f64_f32_past_the_cap",
         ("unpack_xyzir_kernel", None): "test_unpack_xyzir_past_the_cap",
         ("validation_kernel", None): "test_validation_update_past_the_cap",
         ("confusion_kernel", None): "test_confusion_update_past_the_cap"}


def test_every_guarded_kernel_has_a_case():
  """Every __global__ kernel of projection.cu, input_stage.cu, validation.cu and confusion.cu, with every template
  instantiation it is launched with, is declared in CASES (and so launched by a case of this file)."""
  assert source_kernels() == set(CASES)


@pytest.mark.gpu
def test_every_kernel_runs_past_its_cap():
  """Each kernel, launched at the size its case uses, runs with the capped grid (profiler trace), so each case goes
  past its cap; and the declared case sizes exceed each cap at this device's SM count."""
  from tests import test_gpu_cam_pool_input as CP
  sms = _sms()
  lib = _lib.load()
  rp = cap_elems("project_resolve_kernel", sms)
  bt = batch("bench")
  assert bt.total > cap_elems("project_scatter_kernel", sms) and 32 * bt.H * bt.W > rp
  ring = batch("ring")
  assert ring.total > cap_elems("project_scatter_kernel", sms) and ring.B * ring.H * ring.W > rp
  assert input_stage_sizes(sms)[-1] > cap_elems("input_stage_kernel", sms)
  assert all(n > cap_elems("validation_kernel", sms) for n, _ in _validation_case_sizes(sms).values())
  assert all(n > cap_elems("confusion_kernel", sms) for n, _, _ in confusion_cases(sms).values())
  n_is = input_stage_sizes(sms)[-1]
  n_val, nc_val = _validation_case_sizes(sms)["4cap-32"]
  n_cm, nc_cm, _ = confusion_cases(sms)["64x64x2048-32"]
  n_cast = 2 * cap_elems("cast_f64_f32_kernel", sms) + 3
  n_up = 2 * cap_elems("unpack_xyzir_kernel", sms) + 1
  z = lambda *shape, dt=torch.float32: torch.zeros(shape, dtype=dt, device="cuda")
  buf = {"keys": z(bt.B, bt.H, bt.W, dt=torch.int64), "img": z(32, bt.H, bt.W, 6), "in8": z(32, bt.H, bt.W, 8,
         dt=torch.int16), "m8": z(32, bt.H, bt.W, dt=torch.uint8), "is": z(n_is, 6), "lid": z(n_is, 6),
         "probs": z(n_val, nc_val), "lab": z(max(n_val, n_cm), dt=torch.int32), "acc": z(2, dt=torch.float64),
         "cmw": z(nc_val * nc_val, dt=torch.float64), "cm": z(nc_cm * nc_cm, dt=torch.int64),
         "f64": z(n_cast, dt=torch.float64), "f32": z(n_cast), "rec": z(n_up, 5), "p4": z(n_up, 4),
         "ring": z(n_up, dt=torch.int32)}
  p = {k: v.data_ptr() for k, v in buf.items()}

  def launches():
    _lib.check(lib.pcls_project_scatter(bt.d_pts.data_ptr(), None, bt.d_off.data_ptr(), bt.B, bt.total, bt.H, bt.W,
                                        bt.fu, bt.fd, p["keys"], None, None, None, _s()))
    _lib.check(lib.pcls_project_resolve(bt.d_pts.data_ptr(), None, bt.d_off.data_ptr(), 32, bt.H, bt.W, p["keys"],
                                        None, 0, 0.0, p["img"], None, None, _s()))
    for prec in PREC.values():
      _lib.check(lib.pcls_project_resolve_net_input(bt.d_pts.data_ptr(), bt.d_off.data_ptr(), 32, bt.H, bt.W,
                                                    p["keys"], _dbl(KITTI_MEAN), _dbl(KITTI_STD), prec, p["in8"],
                                                    p["m8"], None, _s()))
    _lib.check(lib.pcls_input_stage(p["is"], 6, n_is, _dbl(KITTI_MEAN), _dbl(KITTI_STD), 0, p["lid"], None, None,
                                    None, 0, None, _s()))
    _lib.check(lib.pcls_cast_f64_f32(p["f64"], p["f32"], n_cast, _s()))
    _lib.check(lib.pcls_unpack_xyzir(p["rec"], n_up, p["p4"], p["ring"], _s()))
    _lib.check(lib.pcls_validation_update(p["probs"], p["lab"], p["lab"], None, None, n_val, nc_val, 1, 1e-12, 2.0,
                                          p["acc"], p["cmw"], None, _s()))
    _lib.check(lib.pcls_confusion_update(p["lab"], p["lab"], n_cm, nc_cm, p["cm"], None, _s()))

  def twice():
    # launched straight after the profiler starts, the first kernels can fall before its trace window: wait, then
    # launch every kernel twice; each must be recorded at least once
    time.sleep(0.2)
    launches()
    launches()

  trace = CP._trace(twice)
  seen = set()
  for name, grid in trace:
    m = re.search(r"pcls::(\w+_kernel)(?:<([\w:]+)>)?", name)
    assert m and (m.group(1), m.group(2)) in CASES, name
    key = (m.group(1), m.group(2))
    assert grid[0] == cap_grid(key[0], sms) and grid[1] == grid[2] == 1, (name, grid, cap_grid(key[0], sms))
    seen.add(key)
  assert seen == set(CASES), set(CASES) - seen
