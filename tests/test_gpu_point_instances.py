"""Instance ids on the GPU (pcls_point_instances, ScanSegmenter / ScanEvaluator / segment_scans --instances): exact
(==) against the numpy oracle (oracle/point_instances.py) fed with the device's own scatter outputs and the same point
labels, so every comparison isolates the new kernels.  Every call also checks the guard bands around the outputs and the
scratch, that a sentinel prefill does not survive, and that a second run gives the same bits."""
import itertools
import os

import numpy as np
import pytest
import torch

from oracle import point_instances as PI
from tests.util import synth_scan

pytestmark = pytest.mark.gpu

GUARD = 0x5A5A5A5A      # guard band around instances / instance_counts: must stay untouched
SENTINEL = -12345       # prefill of the outputs: must not survive
KITTI_THINGS = 0b111111110
NC_MASKS = {11: 0b1111100000, 20: KITTI_THINGS, 32: 0x8F0F00F6}


def _lib():
  from pclsegmentation_b200 import _lib
  return _lib


# ---- scan generators ----

def planted_scan(rng, n, nc=20, things=(1, 2, 3, 4, 5, 6, 7, 8), grid=0.0, n_objects=24, seam=True):
  """Synthetic scan with planted objects: boxes and cylinders of thing points at 5-60 m (one across the azimuth seam,
  yaw = +-pi), plus ground and background points of stuff classes.  Labels come from the planted truth.  ``grid`` > 0
  rounds x, y, z to that grid, so that distances equal to tau occur.  Returns (points [n,4] f32, labels [n] i32,
  instance ids [n] i32, 0 = not an object)."""
  stuff = [c for c in range(nc) if c not in things]
  per = np.maximum(rng.multinomial(n // 3, np.ones(n_objects) / n_objects), 1)
  n_obj = int(per.sum())
  pts, lab, inst = [], [], []
  for o, m in enumerate(per):
    r = rng.uniform(5, 60)
    yaw = np.pi if (seam and o == 0) else rng.uniform(-np.pi, np.pi)
    cx, cy = r * np.cos(yaw), r * np.sin(yaw)
    if o % 2 == 0:                                       # box, car-sized
      sx, sy, sz = rng.uniform(1.5, 4.5), rng.uniform(1.5, 2.0), rng.uniform(1.2, 1.8)
      p = (rng.random((m, 3)) - 0.5) * [sx, sy, sz]
    else:                                                # cylinder, person-sized
      a, h, rad = rng.uniform(0, 2 * np.pi, m), rng.uniform(-0.9, 0.9, m), rng.uniform(0.2, 0.4)
      p = np.stack([rad * np.cos(a), rad * np.sin(a), h], 1)
    p = p + [cx, cy, -0.8]
    pts.append(p)
    lab.append(np.full(m, things[o % len(things)]))
    inst.append(np.full(m, o + 1))
  n_rest = n - n_obj
  n_ground = n_rest // 2
  r = rng.uniform(3, 60, n_ground)
  a = rng.uniform(-np.pi, np.pi, n_ground)
  pts.append(np.stack([r * np.cos(a), r * np.sin(a), np.full(n_ground, -1.7) + rng.normal(0, 0.02, n_ground)], 1))
  lab.append(np.full(n_ground, stuff[0]))
  inst.append(np.zeros(n_ground, np.int64))
  bg = synth_scan(rng, n_rest - n_ground)[:, :3]
  pts.append(bg)
  lab.append(rng.choice(stuff, bg.shape[0]))
  inst.append(np.zeros(bg.shape[0], np.int64))
  xyz = np.concatenate(pts)
  if grid > 0:
    xyz = np.round(xyz / grid) * grid
  perm = rng.permutation(n)                              # points in random order, like the other synthetic scans
  out = np.concatenate([xyz, rng.random((n, 1))], 1).astype(np.float32)[perm]
  return out, np.concatenate(lab).astype(np.int32)[perm], np.concatenate(inst).astype(np.int32)[perm]


def bench_scans(B=64):
  """The benchmark batch: 64 scans of 115-125 k points, planted objects, 2 mm grid (tools/point_instances_bench.py)."""
  rng = np.random.default_rng(20261021)
  sizes = rng.integers(115000, 125001, B)
  scans = [planted_scan(rng, int(n), grid=0.002) for n in sizes]
  return sizes, [s[0] for s in scans], [s[1] for s in scans], [s[2] for s in scans]


def keys_vectorised(px, py, rng_val, offsets, B, H, W):
  """Winner keys by the scatter's rule (nearest, then lowest index) for hand-made pixel assignments, vectorised."""
  px, py = np.asarray(px, np.int64), np.asarray(py, np.int64)
  keys = np.full(B * H * W, np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64)
  scan = np.repeat(np.arange(B), np.diff(offsets))
  ok = px >= 0
  local = np.arange(px.size) - np.asarray(offsets)[scan]
  k = (np.asarray(rng_val, np.float32).view(np.uint32).astype(np.uint64) << np.uint64(32)) | local.astype(np.uint64)
  pix = (scan * H + py) * W + px
  np.minimum.at(keys, pix[ok], k[ok])
  return keys.reshape(B, H, W).view(np.int64)


# ---- the device call, with its checks ----

def device_instances(pts, keys, offsets, px, py, labels, nc, mask, ry, rx, wrap, tau, min_points):
  """pcls_point_instances with instances / instance_counts inside guard bands (prefilled with a sentinel) and the scratch
  inside a guard band; checks the bands, that every output was written, and that a second run is bit-identical."""
  lib = _lib()
  L = lib.load()
  B, H, W = keys.shape
  total = int(px.numel())
  nbytes = L.pcls_point_instances_scratch_bytes(B, H, W)
  assert nbytes == 24 * B * H * W
  g = 64
  runs = []
  for _ in range(2):
    out = torch.full((total + 2 * g,), SENTINEL, dtype=torch.int32, device="cuda")
    cnt = torch.full((B + 2 * g,), SENTINEL, dtype=torch.int32, device="cuda")
    for t, n in ((out, total), (cnt, B)):
      t[:g] = GUARD
      t[g + n:] = GUARD
    sbuf = torch.full((nbytes + 2 * 256,), 0xA5, dtype=torch.uint8, device="cuda")
    scratch = sbuf[256:256 + nbytes]
    lib.check(L.pcls_point_instances(pts.data_ptr(), keys.data_ptr(), offsets.data_ptr(), B, H, W, total,
                                     px.data_ptr(), py.data_ptr(), labels.data_ptr(), nc, mask, ry, rx, wrap, tau,
                                     min_points, scratch.data_ptr(), out.data_ptr() + 4 * g, cnt.data_ptr() + 4 * g,
                                     torch.cuda.current_stream().cuda_stream), "pcls_point_instances")
    o, c, s = out.cpu().numpy(), cnt.cpu().numpy(), sbuf.cpu().numpy()
    for a, n, what in ((o, total, "instances"), (c, B, "instance_counts")):
      assert (a[:g] == GUARD).all() and (a[g + n:] == GUARD).all(), "guard band of %s written" % what
      assert not (a[g:g + n] == SENTINEL).any(), "an entry of %s was not written" % what
    assert (s[:256] == 0xA5).all() and (s[256 + nbytes:] == 0xA5).all(), "scratch guard band written"
    runs.append((o[g:g + total].copy(), c[g:g + B].copy()))
  assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1]), "two runs differ"
  return runs[0]


def oracle_instances(pts, keys, offsets, px, py, labels, mask, ry, rx, wrap, tau, min_points):
  c = lambda t: t.cpu().numpy() if torch.is_tensor(t) else t
  return PI.point_instances(c(pts), c(keys), c(offsets), c(px), c(py), c(labels), mask, ry, rx, bool(wrap), tau,
                            min_points)


def check(d, nc, mask, ry, rx, wrap, tau, mp, labels=None):
  lab = d["labels"] if labels is None else labels
  got, cnt = device_instances(d["pts"], d["keys"], d["offsets"], d["px"], d["py"], lab, nc, mask, ry, rx, wrap, tau, mp)
  want, wcnt = oracle_instances(d["pts"], d["keys"], d["offsets"], d["px"], d["py"], lab, mask, ry, rx, wrap, tau, mp)
  bad = np.flatnonzero(got != want)
  assert bad.size == 0, (nc, hex(mask), ry, rx, wrap, tau, mp, bad[:10], got[bad[:10]], want[bad[:10]])
  assert np.array_equal(cnt, wcnt), (cnt, wcnt)
  return got, cnt


def scatter(points, offsets, ring=None, H=64, W=512, fov_up=3.0, fov_down=-25.0):
  from pclsegmentation_b200.laserscan import SphericalProjector
  proj = SphericalProjector(H, W, fov_up, fov_down)
  return proj.project(points, offsets, ring=ring, want_image=False, want_idx=False, want_point_outputs=True)


def to_dev(scans, labels, H=64, W=512, ring=None, **kw):
  sizes = [s.shape[0] for s in scans]
  offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  pts = torch.from_numpy(np.concatenate(scans) if scans else np.zeros((0, 4), np.float32)).cuda()
  offsets = torch.from_numpy(offsets_np).cuda()
  proj = scatter(pts, offsets, ring=ring, H=H, W=W, **kw)
  return dict(pts=pts, offsets=offsets, keys=proj["keys"], px=proj["proj_x"], py=proj["proj_y"],
              labels=torch.from_numpy(np.concatenate(labels).astype(np.int32)).cuda(), sizes=sizes)


@pytest.fixture(scope="module")
def batch():
  """64 x 512, five scans: two planted scans on a 0.25 m grid (distances equal to tau occur), an empty scan, a one-point
  scan and a planted scan on a 2 mm grid; labels in [0, 20)."""
  rng = np.random.default_rng(20261021)
  a = planted_scan(rng, 30000, grid=0.25)
  b = planted_scan(rng, 20000, grid=0.25, n_objects=40)
  c = planted_scan(rng, 25000, grid=0.002)
  one = (np.array([[10.0, 0.5, -0.5, 0.3]], np.float32), np.array([1], np.int32))
  scans = [a[0], np.zeros((0, 4), np.float32), one[0], b[0], c[0]]
  labels = [a[1], np.zeros(0, np.int32), one[1], b[1], c[1]]
  return to_dev(scans, labels)


def _cases():
  """Windows x wrap x tau x min_points, masks cycled over the combinations."""
  windows = [(0, 1), (1, 0), (1, 1), (1, 2), (2, 3), (4, 8)]
  out = []
  for i, ((ry, rx), wrap, tau) in enumerate(itertools.product(windows, (1, 0), (0.2, 0.5, 2.0, 1e4))):
    mp = (1, 2, 10)[i % 3]
    mask = (KITTI_THINGS, 0xFFFFF, 0b10)[(i // 3) % 3]
    out.append((ry, rx, wrap, tau, mp, mask))
  return out


@pytest.mark.parametrize("window", [(0, 1), (1, 0), (1, 1), (1, 2), (2, 3), (4, 8)])
def test_kernel_equals_oracle(batch, window):
  n = 0
  for ry, rx, wrap, tau, mp, mask in _cases():
    if (ry, rx) != window:
      continue
    got, cnt = check(batch, 20, mask, ry, rx, wrap, tau, mp)
    n += 1
    if tau == 0.5 and mask == KITTI_THINGS:
      assert cnt[0] > 5 and cnt[1] == 0, cnt             # objects found; the empty scan has none
  assert n == 8


def test_distances_equal_to_tau_occur_on_the_device(batch):
  """On the 0.25 m grid, node pairs at d^2 == tau^2 exist in the window at tau 0.5, so '<=' vs '<' matters."""
  keys = batch["keys"][0].cpu().numpy().view(np.uint64)
  lo, hi = 0, batch["sizes"][0]
  pts = batch["pts"][lo:hi].cpu().numpy()
  lab = batch["labels"][lo:hi].cpu().numpy()
  occ = keys != PI.EMPTY
  win = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)
  xyz = np.where(occ[..., None], pts[np.where(occ, win, 0)][..., :3], 0)
  thing = occ & (((KITTI_THINGS >> np.where(occ, lab[np.where(occ, win, 0)], 0)) & 1) == 1)
  eq = thing[:, :-1] & thing[:, 1:] & (PI.dist2(xyz[:, :-1], xyz[:, 1:]) == np.float32(0.25))
  assert eq.sum() > 10
  # and the boundary changes the answer: the kernel agrees with the oracle both at tau 0.5 and one ulp below
  below = float(np.nextafter(np.float32(0.5), np.float32(0)))
  a, _ = check(batch, 20, KITTI_THINGS, 0, 1, 1, 0.5, 1)
  b, _ = check(batch, 20, KITTI_THINGS, 0, 1, 1, below, 1)
  assert not np.array_equal(a, b)


@pytest.mark.parametrize("mp", ["boundary", "boundary-1"])
def test_min_points_at_the_exact_boundary(batch, mp):
  want, _ = oracle_instances(batch["pts"], batch["keys"], batch["offsets"], batch["px"], batch["py"], batch["labels"],
                             KITTI_THINGS, 1, 2, 1, 0.5, 1)
  sizes = np.bincount(want[want > 0])
  size = int(np.median(sizes[sizes > 3]))                  # a component size that occurs
  check(batch, 20, KITTI_THINGS, 1, 2, 1, 0.5, size if mp == "boundary" else size + 1)


@pytest.mark.parametrize("nc", [11, 20, 32])
def test_class_counts_and_masks(nc):
  rng = np.random.default_rng(nc)
  things = [c for c in range(nc) if (NC_MASKS[nc] >> c) & 1]
  scans = [planted_scan(rng, 15000, nc=nc, things=things, grid=0.25) for _ in range(3)]
  d = to_dev([s[0] for s in scans], [s[1] for s in scans])
  for mask in (NC_MASKS[nc], 0, (1 << nc) - 1 if nc < 32 else 0xFFFFFFFF):
    got, cnt = check(d, nc, mask, 1, 2, 1, 0.5, 3)
    if mask == 0:
      assert not got.any() and not cnt.any()


def hand_batch(B, H, W, px, py, xyz, labels, rng_val=None):
  n = px.size
  offsets_np = np.linspace(0, n, B + 1).astype(np.int64) if B > 1 else np.array([0, n], np.int64)
  rng_val = np.ones(n, np.float32) if rng_val is None else rng_val
  keys = keys_vectorised(px, py, rng_val, offsets_np, B, H, W)
  pts = np.concatenate([np.asarray(xyz, np.float32), np.zeros((n, 1), np.float32)], 1)
  return dict(pts=torch.from_numpy(pts).cuda(), offsets=torch.from_numpy(offsets_np).cuda(),
              keys=torch.from_numpy(keys).cuda(), px=torch.from_numpy(px.astype(np.int32)).cuda(),
              py=torch.from_numpy(py.astype(np.int32)).cuda(),
              labels=torch.from_numpy(np.asarray(labels, np.int32)).cuda(), sizes=[n])


def test_objects_exactly_tau_apart_and_touching_objects_of_different_classes():
  # row 5: class 1 at columns 10-13 and class 1 at 14-17, 0.5 m (== tau) between columns 13 and 14: one object;
  # row 9: class 1 at 10-13 touching class 2 at 14-17: two objects; row 20: the gap one float32 ulp above tau: two
  x = np.float32(0.125) * np.arange(8, dtype=np.float32)       # 0 .. 0.875, 0.125 apart
  gaps = {5: x + np.where(np.arange(8) >= 4, np.float32(0.375), np.float32(0)),
          9: x - np.where(np.arange(8) >= 4, np.float32(0.125), np.float32(0)),
          20: x + np.where(np.arange(8) >= 4, np.float32(0.375), np.float32(0))}
  gaps[20][4] = np.nextafter(gaps[20][4], np.float32(2))
  px, py, xyz, lab = [], [], [], []
  for row, l2 in ((5, 1), (9, 2), (20, 1)):
    for k in range(8):
      px.append(10 + k)
      py.append(row)
      xyz.append([gaps[row][k], float(row), 0.0])
      lab.append(1 if k < 4 else l2)
  assert PI.dist2(xyz[3], xyz[4]) == np.float32(0.25) and PI.dist2(xyz[19], xyz[20]) > np.float32(0.25)
  d = hand_batch(1, 32, 64, np.array(px), np.array(py), xyz, lab)
  got, cnt = check(d, 20, KITTI_THINGS, 1, 2, 1, 0.5, 1)
  assert cnt.tolist() == [5]
  assert got.tolist() == [1] * 8 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4


def test_ring_around_all_columns_is_one_component_through_the_seam():
  H, W = 64, 2048
  c = np.arange(W)
  a = 2 * np.pi * (c + 0.5) / W
  # a ring of radius 20 m (6 cm between columns) that climbs 1 mm per column from column 1000 on, around the seam, back
  # to column 999: one cut, between 999 and 1000 (2 m); columns W-1 and 0 are 1 mm apart in height
  z = 0.001 * ((c - 1000) % W)
  xyz = np.stack([20 * np.cos(a), 20 * np.sin(a), z], 1)
  d = hand_batch(1, H, W, c, np.full(W, 40), xyz, np.full(W, 3))
  got, cnt = check(d, 20, KITTI_THINGS, 0, 1, 1, 0.5, 1)
  assert cnt.tolist() == [1] and (got == 1).all()              # joined through the seam
  got, cnt = check(d, 20, KITTI_THINGS, 0, 1, 0, 0.5, 1)
  assert cnt.tolist() == [2] and (got[:1000] == 1).all() and (got[1000:] == 2).all()


def test_serpentine_component_through_every_row():
  """A path through every pixel, row by row in alternating directions: neighbours in the window are far apart except
  along the path, so the union-find trees are deep."""
  H, W = 64, 2048
  r = np.repeat(np.arange(H), W)
  c = np.tile(np.arange(W), H)
  c = np.where(r % 2 == 0, c, W - 1 - c)
  s = np.arange(H * W, dtype=np.float64)                    # position along the path
  xyz = np.stack([0.25 * s, np.zeros_like(s), np.zeros_like(s)], 1)
  perm = np.random.default_rng(1).permutation(H * W)
  d = hand_batch(1, H, W, c[perm], r[perm], xyz[perm], np.full(H * W, 2))
  got, cnt = check(d, 20, KITTI_THINGS, 1, 2, 1, 0.3, 1)
  assert cnt.tolist() == [1] and (got == 1).all()
  # every 100th step 0.5 m long: 1310 components, numbered along the path's pixels
  xyz2 = np.stack([0.25 * s + 0.25 * (s // 100), np.zeros_like(s), np.zeros_like(s)], 1)
  d = hand_batch(1, H, W, c[perm], r[perm], xyz2[perm], np.full(H * W, 2))
  got, cnt = check(d, 20, KITTI_THINGS, 1, 2, 1, 0.3, 1)
  assert cnt[0] > 1000


def test_all_thing_image_is_one_component():
  H, W = 64, 2048
  r = np.repeat(np.arange(H), W)
  c = np.tile(np.arange(W), H)
  xyz = np.stack([0.01 * c, 0.01 * r, np.zeros(H * W)], 1)
  rng = np.random.default_rng(2)
  # two points per pixel: winners and near losers of the same class, so sizes count 2 per pixel
  px, py = np.concatenate([c, c]), np.concatenate([r, r])
  rv = np.concatenate([np.full(H * W, 5.0), np.full(H * W, 6.0)]).astype(np.float32)
  xyz2 = np.concatenate([xyz, xyz + [0, 0, 0.1]])
  perm = rng.permutation(2 * H * W)
  d = hand_batch(1, H, W, px[perm], py[perm], xyz2[perm], np.full(2 * H * W, 4), rng_val=rv[perm])
  got, cnt = check(d, 20, KITTI_THINGS, 1, 2, 1, 0.5, 2 * H * W)
  assert cnt.tolist() == [1] and (got == 1).all()
  got, cnt = check(d, 20, KITTI_THINGS, 1, 2, 1, 0.5, 2 * H * W + 1)
  assert cnt.tolist() == [0] and (got == 0).all()


def test_ring_projection_keys():
  """Ring projection: the keys carry ~index, not the depth; the winner is still found through the low word."""
  rng = np.random.default_rng(5)
  Hr, Wr = 32, 256
  scans = [planted_scan(rng, 12000, grid=0.25), planted_scan(rng, 7000, grid=0.25)]
  rings = [rng.integers(0, Hr, s[0].shape[0]).astype(np.int32) for s in scans]
  d = to_dev([s[0] for s in scans], [s[1] for s in scans], H=Hr, W=Wr,
             ring=torch.from_numpy(np.concatenate(rings)).cuda(), fov_up=10.0, fov_down=-30.0)
  keys = d["keys"].cpu().numpy().view(np.uint64)
  assert ((keys[keys != PI.EMPTY] >> np.uint64(32)) > np.uint64(0x80000000)).all()     # ~index in the high word
  for ry, rx, wrap, tau in ((1, 2, 1, 0.5), (2, 3, 0, 2.0)):
    check(d, 20, KITTI_THINGS, ry, rx, wrap, tau, 2)


def test_benchmark_batch_against_oracle():
  """The 64-scan benchmark batch at 64 x 2048 with the planted labels, default Clustering parameters."""
  sizes, scans, labels, _ = bench_scans()
  d = to_dev(scans, labels, H=64, W=2048)
  got, cnt = check(d, 20, KITTI_THINGS, 1, 2, 1, 0.5, 10)
  assert (cnt > 10).all()


# ---- pipeline ----

@pytest.fixture(scope="module")
def small_model():
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map["squeezesegv2kitti"]()
  mc.AZIMUTH_LEVEL = 512
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(2)
  return mc, model


def test_segment_device_equals_the_direct_call(small_model):
  from pclsegmentation_b200.pipeline import KNN, Clustering, ScanSegmenter
  mc, model = small_model
  rng = np.random.default_rng(8)
  scans = [planted_scan(rng, n, grid=0.002)[0] for n in (20000, 15000)] + [np.zeros((0, 4), np.float32)]
  sizes = [s.shape[0] for s in scans]
  pts = torch.from_numpy(np.concatenate(scans)).cuda()
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).cuda()
  seg = ScanSegmenter(model, 3.0, -25.0)
  with pytest.raises(ValueError):
    seg.segment_device(pts, offsets, instances=Clustering())
  # a thing set that the random-init network predicts: its two most frequent classes
  base = seg.segment_device(pts, offsets, want_point_labels=True, knn=KNN())
  assert "instances" not in base
  freq = np.bincount(base["point_labels"].cpu().numpy(), minlength=mc.NUM_CLASS)
  things = [int(c) for c in np.argsort(-freq)[:2]]
  cl = Clustering(tau=2.0, rows=1, cols=3, min_points=2, thing_classes=things)
  one = seg.segment_device(pts, offsets, want_point_labels=True, knn=KNN(), instances=cl)
  two = seg.segment_device(pts, offsets, want_point_labels=True, knn=KNN(), instances=cl, want_image=True)
  assert torch.equal(one["point_labels"], base["point_labels"]) and torch.equal(one["predictions"], base["predictions"])
  assert torch.equal(one["instances"], two["instances"]) and torch.equal(one["instance_counts"],
                                                                         two["instance_counts"])
  proj = scatter(pts, offsets)
  d = dict(pts=pts, offsets=offsets, keys=proj["keys"], px=proj["proj_x"], py=proj["proj_y"],
           labels=one["point_labels"])
  got, cnt = check(d, mc.NUM_CLASS, cl.thing_mask(mc), 1, 3, 1, 2.0, 2)
  assert np.array_equal(one["instances"].cpu().numpy(), got) and np.array_equal(one["instance_counts"].cpu().numpy(), cnt)
  assert cnt[0] > 0 and cnt[2] == 0
  words = seg.label_words(one, sizes)
  inst = one["instances"].cpu().numpy()
  lab = one["point_labels"].cpu().numpy()
  assert np.array_equal(np.concatenate(words), (inst.astype(np.uint32) << 16) | lab.astype(np.uint32))
  inv = np.arange(mc.NUM_CLASS, dtype=np.uint32) * 3 + 1
  assert np.array_equal(np.concatenate(seg.label_words(one, sizes, inv)) & 0xFFFF, inv[lab])
  assert np.array_equal(np.concatenate(seg.label_words(base, sizes)), lab.astype(np.uint32))
  fake = dict(one, instances=torch.full_like(one["instances"], 0x10000))
  with pytest.raises(ValueError):
    seg.label_words(fake, sizes)


def _write_planted_dataset(tmp_path, rng, sizes, lab_of_class):
  scan_dir, lab_dir = tmp_path / "velodyne", tmp_path / "labels"
  scan_dir.mkdir()
  lab_dir.mkdir()
  words = []
  for i, n in enumerate(sizes):
    pts, lab, inst = planted_scan(rng, n, grid=0.002)
    pts.tofile(str(scan_dir / ("%06d.bin" % i)))
    w = (inst.astype(np.uint32) << 16) | lab_of_class[lab].astype(np.uint32)
    w.tofile(str(lab_dir / ("%06d.label" % i)))
    words.append(w)
  return scan_dir, lab_dir, words


def test_segment_scans_instances_cli(tmp_path, capsys):
  import yaml
  from pclsegmentation_b200 import segment_scans
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader, learning_map_lut
  from pclsegmentation_b200.metrics import PanopticQuality
  from pclsegmentation_b200.pipeline import KNN, Clustering, ScanSegmenter
  from pclsegmentation_b200.utils.args_loader import load_model_config
  rng = np.random.default_rng(12)
  sizes = [8000, 6000, 7000]
  raw_of_class = np.array([0, 10, 11, 15, 18, 20, 30, 31, 32, 40, 44, 48, 49, 50, 51, 70, 71, 72, 80, 81], np.uint32)
  scan_dir, lab_dir, words = _write_planted_dataset(tmp_path, rng, sizes, raw_of_class)
  learning_map = {int(r): c for c, r in enumerate(raw_of_class)}
  learning_map_inv = {c: int(r) for c, r in enumerate(raw_of_class)}
  ypath = tmp_path / "map.yaml"
  ypath.write_text(yaml.safe_dump({"learning_map": learning_map, "learning_map_inv": learning_map_inv}))
  base = ["--scans", str(scan_dir / "*.bin"), "--format", "kitti", "-m", "squeezesegv2", "-n", "squeezesegv2kitti",
          "--random_init", "--batch", "2", "--learning_map", str(ypath)]
  segment_scans.main(base + ["--output_dir", str(tmp_path / "sem")])
  clus = ["--instances", "--cluster_tau", "1.0", "--min_points", "3"]
  capsys.readouterr()
  rep = segment_scans.main(base + clus + ["--output_dir", str(tmp_path / "pan"), "--labels", str(lab_dir / "*.label")])
  printed = capsys.readouterr().out
  files = sorted(str(p) for p in scan_dir.iterdir())
  names = [os.path.splitext(os.path.basename(f))[0] + ".label" for f in files]
  # the lower 16 bits are byte-identical to the run without --instances
  sem = [np.fromfile(str(tmp_path / "sem" / n), np.uint32) for n in names]
  pan = [np.fromfile(str(tmp_path / "pan" / n), np.uint32) for n in names]
  for s, p in zip(sem, pan):
    assert np.array_equal(p & 0xFFFF, s) and p.dtype == np.uint32
  assert any((p >> 16).any() for p in pan), "no instance was written"
  # the upper 16 bits are the device instances; the report is PanopticQuality fed by the oracle
  mc, model = load_model_config("squeezesegv2", "squeezesegv2kitti")     # the CLI's model: same seeded init
  seg = ScanSegmenter(model, 3.0, -25.0)
  cl = Clustering(tau=1.0, min_points=3)
  loader = ScanBatchLoader("kitti")
  lut = learning_map_lut(learning_map)
  pq = PanopticQuality(mc.NUM_CLASS, cl.thing_ids(mc), mc.CLASSES.index("None"))
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2])
    res = seg.segment_device(data["points"], data["offsets"], want_point_labels=True, knn=KNN(), instances=cl)
    proj = scatter(data["points"], data["offsets"], H=mc.ZENITH_LEVEL, W=mc.AZIMUTH_LEVEL)   # the CLI's 64 x 1024
    want, _ = oracle_instances(data["points"], proj["keys"], data["offsets"], proj["proj_x"], proj["proj_y"],
                               res["point_labels"], cl.thing_mask(mc), 1, 2, 1, 1.0, 3)
    assert np.array_equal(res["instances"].cpu().numpy(), want)
    offs = data["offsets"].cpu().numpy()
    lab = res["point_labels"].cpu().numpy()
    for j, n in enumerate(names[lo:lo + 2]):
      sl = slice(offs[j], offs[j + 1])
      assert np.array_equal(pan[lo + j] >> 16, want[sl].astype(np.uint32))
      w = words[lo + j]
      pq.update(lut[w & 0xFFFF], w >> 16, lab[sl], want[sl])
  r = pq.result()
  for key in ("tp", "fp", "fn", "pq", "sq", "rq"):
    assert np.array_equal(rep["panoptic"][key], r[key]), key
  assert rep["panoptic"]["pq_mean"] == r["pq_mean"]
  assert "PANOPTIC" in printed and "PQ: {} ".format(r["pq_mean"]) in printed and "CAR PQ:" in printed
  assert r["fn"].sum() > 0


def test_segment_scans_instances_nuscenes_skips_the_report(tmp_path, capsys):
  from pclsegmentation_b200 import segment_scans
  rng = np.random.default_rng(13)
  scan_dir, lab_dir = tmp_path / "velodyne", tmp_path / "labels"
  scan_dir.mkdir()
  lab_dir.mkdir()
  for i, n in enumerate((5000, 4000)):
    pts, lab, _ = planted_scan(rng, n, nc=11, things=(5, 6, 7, 8, 9), grid=0.002)
    rec = np.concatenate([pts, rng.integers(0, 32, (n, 1)).astype(np.float32)], 1)
    rec.astype(np.float32).tofile(str(scan_dir / ("%06d.bin" % i)))
    lab.astype(np.uint8).tofile(str(lab_dir / ("%06d.bin" % i)))
  args = ["--scans", str(scan_dir / "*.bin"), "--format", "nuscenes", "-m", "squeezesegv2", "-n", "squeezesegv2",
          "--random_init", "--output_dir", str(tmp_path / "out"), "--instances", "--labels", str(lab_dir / "*.bin")]
  capsys.readouterr()
  segment_scans.main(args)
  printed = capsys.readouterr().out
  assert "MIoU" in printed and "no panoptic report" in printed and "PANOPTIC" not in printed
  out = np.fromfile(str(tmp_path / "out" / "000000.label"), np.uint32)
  assert out.shape == (5000,)
