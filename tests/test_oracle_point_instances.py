"""Instance ids (pcls_point_instances) and panoptic quality: hand-built cases that pin each rule of the contract on the
numpy oracle, the oracle against a plain union-find, PanopticQuality against hand cases and a brute-force per-pair loop,
and the argument checks of the C entry points, which run before any CUDA call (no GPU needed)."""
import ctypes

import numpy as np
import pytest

from oracle import point_instances as PI
from pclsegmentation_b200 import _lib

H, W = 4, 16
THING = 0b0110          # classes 1 and 2 are things, 0 and 3 stuff


def run(pts, thing=THING, ry=1, rx=2, wrap=True, tau=0.5, min_points=1, Hh=H, Ww=W):
  """pts: list of (row, col, x, y, z, label, range); row -1 = dropped.  One scan -> (instances, count)."""
  a = np.array(pts, np.float64).reshape(-1, 7)
  py, px = a[:, 0].astype(np.int64), a[:, 1].astype(np.int64)
  px[py < 0] = -1
  xyz = np.concatenate([a[:, 2:5], np.zeros((a.shape[0], 1))], 1).astype(np.float32)
  keys = PI.keys_from_pixels(px, py, a[:, 6].astype(np.float32), [0, a.shape[0]], Hh, Ww)
  out, counts = PI.point_instances(xyz, keys, [0, a.shape[0]], px, py, a[:, 5].astype(np.int64), thing, ry, rx, wrap,
                                   tau, min_points)
  return out.tolist(), int(counts[0])


def test_distance_equal_to_tau_joins_and_one_ulp_above_does_not():
  assert run([(0, 0, 0.0, 0, 0, 1, 5), (0, 1, 0.5, 0, 0, 1, 5)]) == ([1, 1], 1)
  above = float(np.nextafter(np.float32(0.5), np.float32(1)))
  assert PI.dist2([above, 0, 0], [0, 0, 0]) > np.float32(0.25)
  assert run([(0, 0, 0.0, 0, 0, 1, 5), (0, 1, above, 0, 0, 1, 5)]) == ([1, 2], 2)
  # tau^2 is rounded once to float32: tau 0.1 -> fl32(0.1 * 0.1)
  t2 = np.float32(np.float32(0.1) * np.float32(0.1))
  assert run([(0, 0, 0, 0, 0, 1, 5), (0, 1, 0, 0, 0.1, 1, 5)], tau=0.1)[1] == (1 if PI.dist2([0, 0, 0.1], [0, 0, 0]) <= t2
                                                                             else 2)


def test_window_edges_in_rows_and_columns():
  near = lambda r, c: (r, c, 0.01 * r, 0.01 * c, 0, 1, 5)
  assert run([near(0, 5), near(1, 5)], ry=1, rx=0)[1] == 1
  assert run([near(0, 5), near(2, 5)], ry=1, rx=0)[1] == 2
  assert run([near(0, 5), near(2, 5)], ry=2, rx=0)[1] == 1
  assert run([near(0, 5), near(0, 7)], ry=0, rx=2)[1] == 1
  assert run([near(0, 5), near(0, 8)], ry=0, rx=2)[1] == 2
  assert run([near(0, 5), near(1, 3)], ry=1, rx=2)[1] == 1     # diagonal corner of the window
  assert run([near(0, 5), near(1, 2)], ry=1, rx=2)[1] == 2
  assert run([near(1, 5), near(0, 7)], ry=1, rx=2)[1] == 1     # the other diagonal: the pair from the lower row
  assert run([near(0, 5), near(0, 6)], ry=1, rx=0)[1] == 2     # rx 0: no column neighbour at all


def test_wrap_joins_columns_0_and_w_minus_1():
  pts = [(1, 0, 1.0, 0.0, 0, 2, 5), (1, W - 1, 1.0, 0.05, 0, 2, 5), (2, W - 2, 1.0, 0.1, 0, 2, 5)]
  assert run(pts, wrap=True) == ([1, 1, 1], 1)
  assert run(pts, wrap=False) == ([1, 2, 2], 2)
  # column distance modulo W: W-2 to 1 is 3 > rx 2
  assert run([(0, 1, 0, 0, 0, 1, 5), (0, W - 2, 0, 0, 0, 1, 5)], wrap=True)[1] == 2
  assert run([(0, 0, 0, 0, 0, 1, 5), (0, W - 2, 0, 0, 0, 1, 5)], wrap=True)[1] == 1


def test_the_two_loser_conditions_each_failing_alone():
  win = (0, 3, 1.0, 0, 0, 1, 5)
  same_near = (0, 3, 1.3, 0, 0, 1, 6)
  other_label = (0, 3, 1.1, 0, 0, 2, 6)        # a thing label, but not the winner's
  far = (0, 3, 1.6, 0, 0, 1, 6)                # d 0.6 > tau
  stuff = (0, 3, 1.0, 0, 0, 0, 6)
  assert run([win, same_near, other_label, far, stuff]) == ([1, 1, 0, 0, 0], 1)
  # the loser's distance is measured to the winner, not to the nearest member
  assert run([win, (0, 4, 1.45, 0, 0, 1, 5), (0, 3, 1.6, 0, 0, 1, 6)])[0] == [1, 1, 0]


def test_size_counts_losers_at_the_min_points_boundary():
  pts = [(0, 3, 1.0, 0, 0, 1, 5), (0, 3, 1.1, 0, 0, 1, 6), (0, 3, 1.2, 0, 0, 1, 7), (2, 9, 5, 5, 5, 1, 5)]
  assert run(pts, min_points=3) == ([1, 1, 1, 0], 1)      # size 3 == min_points: kept
  assert run(pts, min_points=4) == ([0, 0, 0, 0], 0)      # one less than min_points: dropped
  assert run(pts, min_points=1) == ([1, 1, 1, 2], 2)


def test_numbering_is_by_smallest_pixel_index_not_point_order():
  # component B (pixels 2*16+10.., min 42) listed first; component A (pixels 5, 6, min 5) last; C at pixel 20
  pts = [(2, 10, 9, 9, 0, 1, 5), (2, 11, 9, 9.1, 0, 1, 5), (1, 4, 4, 4, 0, 2, 5), (0, 6, 0, 0.1, 0, 1, 5),
         (0, 5, 0, 0, 0, 1, 5)]
  assert run(pts) == ([3, 3, 2, 1, 1], 3)
  # a component's id follows its minimum pixel (9), although it reaches past the other component's (17) in pixels
  # (24, 41) and its points come after that component's in point order
  pts = [(1, 1, 5, 5, 0, 1, 5), (2, 9, 0, 0.4, 0, 1, 5), (1, 8, 0, 0.2, 0, 1, 5), (0, 9, 0, 0, 0, 1, 5)]
  assert run(pts) == ([2, 1, 1, 1], 2)


def test_stuff_and_dropped_points_get_zero():
  pts = [(0, 0, 0, 0, 0, 0, 5), (0, 1, 0, 0, 0, 3, 5), (-1, -1, 0, 0, 0, 1, 5), (0, 2, 0, 0, 0, 1, 5)]
  assert run(pts) == ([0, 0, 0, 1], 1)
  assert run(pts, thing=0) == ([0, 0, 0, 0], 0)
  assert run(pts, thing=0xF) == ([1, 2, 0, 3], 3)          # stuff classes made things: different labels never join


def test_empty_scan():
  keys = np.full((1, H, W), -1, np.int64)
  out, counts = PI.point_instances(np.zeros((0, 4), np.float32), keys, [0, 0], np.zeros(0, np.int32),
                                   np.zeros(0, np.int32), np.zeros(0, np.int32), THING)
  assert out.shape == (0,) and counts.tolist() == [0]


def union_find_reference(pts, px, py, labels, keys, thing, ry, rx, wrap, tau, min_points):
  """Independent restatement: pairwise loops over the nodes with a sequential union-find."""
  Hh, Ww = keys.shape
  k = keys.view(np.uint64)
  t2 = np.float32(np.float32(tau) * np.float32(tau))
  nodes = {}
  for r in range(Hh):
    for c in range(Ww):
      if k[r, c] != PI.EMPTY:
        i = int(k[r, c] & np.uint64(0xFFFFFFFF))
        if (thing >> int(labels[i])) & 1:
          nodes[r * Ww + c] = i
  parent = {p: p for p in nodes}

  def find(x):
    while parent[x] != x:
      x = parent[x]
    return x
  for p, i in nodes.items():
    for q, j in nodes.items():
      if q <= p:
        continue
      dr = abs(p // Ww - q // Ww)
      dc = abs(p % Ww - q % Ww)
      if wrap:
        dc = min(dc, Ww - dc)
      if dr <= ry and dc <= rx and labels[i] == labels[j] and PI.dist2(pts[i, :3], pts[j, :3]) <= t2:
        a, b = find(p), find(q)
        parent[max(a, b)] = min(a, b)
  belong = {}
  for n in range(pts.shape[0]):
    if px[n] < 0:
      continue
    p = py[n] * Ww + px[n]
    if p not in nodes:
      continue
    w = nodes[p]
    if n == w or (labels[n] == labels[w] and PI.dist2(pts[n, :3], pts[w, :3]) <= t2):
      belong[n] = find(p)
  sizes = {}
  for r in belong.values():
    sizes[r] = sizes.get(r, 0) + 1
  ids = {r: i + 1 for i, r in enumerate(sorted(r for r, s in sizes.items() if s >= min_points))}
  return [ids.get(belong.get(n, -1), 0) for n in range(pts.shape[0])]


@pytest.mark.parametrize("seed", range(6))
def test_oracle_equals_a_plain_union_find(seed):
  rng = np.random.default_rng(seed)
  Hh, Ww, n = 6, 12, 140
  px = rng.integers(0, Ww, n)
  py = rng.integers(0, Hh, n)
  px[::17] = -1
  py[::17] = -1
  pts = np.zeros((n, 4), np.float32)
  pts[:, :3] = 0.25 * rng.integers(0, 5, (n, 3))
  labels = rng.integers(0, 4, n)
  rng_val = rng.uniform(1, 9, n).astype(np.float32)
  keys = PI.keys_from_pixels(px, py, rng_val, [0, n], Hh, Ww)[0]
  for ry, rx, wrap, tau, mp in ((1, 2, True, 0.5, 1), (0, 1, False, 0.25, 2), (2, 3, True, 0.6, 3), (1, 0, False, 1e4, 1)):
    got, count, _ = PI.scan_instances(pts, keys, px, py, labels, THING, ry, rx, wrap, tau, mp)
    want = union_find_reference(pts, px, py, labels, keys, THING, ry, rx, wrap, tau, mp)
    assert got.tolist() == want, (ry, rx, wrap, tau, mp)
    assert count == max(want)


def test_clustering_thing_classes_resolve_by_name():
  from pclsegmentation_b200.pipeline import Clustering
  from pclsegmentation_b200.utils.args_loader import config_map
  kitti = config_map["squeezesegv2kitti"]()
  assert Clustering().thing_ids(kitti) == list(range(1, 9))
  assert Clustering().thing_mask(kitti) == 0b111111110
  ika = config_map["squeezesegv2"]()
  assert [ika.CLASSES[i] for i in Clustering().thing_ids(ika)] == ["Person", "Two-wheeler", "Car", "Truck", "Bus"]
  dk = config_map["darknet21"]()
  assert [dk.CLASSES[i] for i in Clustering().thing_ids(dk)] == ["Person", "TwoWheeler", "Car", "Truck", "Bus"]
  assert Clustering(thing_classes=["car", 6]).thing_ids(kitti) == [1, 6]
  assert Clustering(thing_classes=[]).thing_mask(kitti) == 0
  with pytest.raises(ValueError):
    Clustering(thing_classes=[20]).thing_ids(kitti)
  c = Clustering()
  assert (c.tau, c.rows, c.cols, c.min_points, c.wrap) == (0.5, 1, 2, 10, True)


# ---- panoptic quality ----

def pq_of(gt_c, gt_i, pr_c, pr_i, things=(1, 2), ignore=0, min_gt=1):
  from pclsegmentation_b200.metrics import PanopticQuality
  m = PanopticQuality(4, things, ignore, min_gt_points=min_gt)
  m.update(gt_c, gt_i, pr_c, pr_i)
  return m


def test_pq_perfect_match():
  gc = [1, 1, 1, 2, 2, 3]
  gi = [5, 5, 5, 9, 9, 0]
  m = pq_of(gc, gi, gc, [1, 1, 1, 2, 2, 0])
  r = m.result()
  assert r["tp"].tolist() == [1, 1] and r["fp"].tolist() == [0, 0] and r["fn"].tolist() == [0, 0]
  assert r["pq"].tolist() == [1.0, 1.0] and r["pq_mean"] == r["sq_mean"] == r["rq_mean"] == 1.0


def test_pq_iou_exactly_half_does_not_match():
  # gt 4 points, prediction covers 2 of them plus nothing else: IoU 2 / 4 = 0.5
  gc, gi = [1, 1, 1, 1], [1, 1, 1, 1]
  r = pq_of(gc, gi, [1, 1, 3, 3], [1, 1, 0, 0]).result()
  assert r["tp"][0] == 0 and r["fp"][0] == 1 and r["fn"][0] == 1 and r["pq"][0] == 0.0
  r = pq_of(gc, gi, [1, 1, 1, 3], [1, 1, 1, 0]).result()          # IoU 3 / 4
  assert r["tp"][0] == 1 and r["fp"][0] == 0 and r["fn"][0] == 0
  assert r["sq"][0] == 0.75 and r["rq"][0] == 1.0 and r["pq"][0] == 0.75


def test_pq_split_and_merge():
  # one object split in two predictions of 3 + 1 points: the larger one matches (IoU 3/4), the other is a FP
  r = pq_of([1] * 4, [1] * 4, [1] * 4, [1, 1, 1, 2]).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (1, 1, 0)
  assert r["pq"][0] == pytest.approx(0.75 / 1.5)
  # two objects (3 and 2 points) merged into one prediction: IoU 3/5 with the first, 2/5 with the second
  r = pq_of([1] * 5, [1, 1, 1, 2, 2], [1] * 5, [7] * 5).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (1, 0, 1)
  assert r["pq"][0] == pytest.approx(0.6 / 1.5)
  # equal halves: IoU 0.5 with each -> no match at all
  r = pq_of([1] * 4, [1, 1, 2, 2], [1] * 4, [3] * 4).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (0, 1, 2)


def test_pq_none_ground_truth_is_removed_first():
  # the prediction covers the gt object (2 points) and 2 points of class None: IoU 1 after removal, 0.5 before
  r = pq_of([1, 1, 0, 0], [1, 1, 0, 0], [1, 1, 1, 1], [1, 1, 1, 1]).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (1, 0, 0) and r["pq"][0] == 1.0
  # a prediction entirely on None points is no segment at all
  r = pq_of([0, 0, 2], [0, 0, 0], [1, 1, 2], [4, 4, 0]).result()
  assert r["fp"].tolist() == [0, 0] and not r["counted"].any() and r["pq_mean"] == 0.0


def test_pq_small_ground_truth_is_ignored():
  # gt segment of 3 points < min_gt 4: neither TP nor FN; a prediction on it (3 of 4 points on it) is no FP
  r = pq_of([1, 1, 1, 1], [1, 1, 1, 0], [1, 1, 1, 1], [2, 2, 2, 2], min_gt=4).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (0, 0, 0) and not r["counted"][0]
  # exactly half of the prediction on the ignored segment: a FP
  r = pq_of([1, 1, 1, 1, 1, 1], [1, 1, 1, 0, 0, 0], [1] * 6, [2] * 6, min_gt=4).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (0, 1, 0)
  # the same object counted (min_gt 3): IoU 3/4 TP
  r = pq_of([1, 1, 1, 1], [1, 1, 1, 0], [1, 1, 1, 1], [2, 2, 2, 2], min_gt=3).result()
  assert (r["tp"][0], r["fp"][0], r["fn"][0]) == (1, 0, 0)


def test_pq_accumulates_over_scans_and_classes():
  from pclsegmentation_b200.metrics import PanopticQuality
  m = PanopticQuality(4, [1, 2], 0, min_gt_points=1)
  m.update([1, 1], [1, 1], [1, 1], [1, 1])               # TP, IoU 1
  m.update([1, 1, 2], [1, 1, 0], [1, 1, 2], [1, 2, 1])   # class 1 split: IoU 0.5 each -> FN + 2 FP; class 2: FP
  r = m.result()
  assert r["tp"].tolist() == [1, 0] and r["fp"].tolist() == [2, 1] and r["fn"].tolist() == [1, 0]
  assert r["pq"][0] == pytest.approx(1.0 / (1 + 1 + 0.5)) and r["pq"][1] == 0.0
  assert r["pq_mean"] == pytest.approx((r["pq"][0] + 0.0) / 2)


def brute_force_pq(scans, things, ignore, min_gt, nc):
  tp, fp, fn, s = np.zeros(nc, int), np.zeros(nc, int), np.zeros(nc, int), np.zeros(nc)
  for gc, gi, pc, pi in scans:
    keep = [n for n in range(len(gc)) if gc[n] != ignore]
    gseg, pseg = {}, {}
    for n in keep:
      if gc[n] in things and gi[n] > 0:
        gseg.setdefault((gc[n], gi[n]), set()).add(n)
      if pc[n] in things and pi[n] > 0:
        pseg.setdefault((pc[n], pi[n]), set()).add(n)
    matched_p = set()
    for gk, g in gseg.items():
      if len(g) < min_gt:
        continue
      hit = None
      for pk, p in pseg.items():
        if pk[0] == gk[0] and len(g & p) / len(g | p) > 0.5:
          hit = pk
          s[gk[0]] += len(g & p) / len(g | p)
      if hit is None:
        fn[gk[0]] += 1
      else:
        tp[gk[0]] += 1
        matched_p.add(hit)
    for pk, p in pseg.items():
      if pk in matched_p:
        continue
      ign = sum(len(g & p) for gk, g in gseg.items() if gk[0] == pk[0] and len(g) < min_gt)
      if not ign > 0.5 * len(p):
        fp[pk[0]] += 1
  return tp, fp, fn, s


@pytest.mark.parametrize("seed", range(5))
def test_pq_equals_a_brute_force_pair_loop(seed):
  from pclsegmentation_b200.metrics import PanopticQuality
  rng = np.random.default_rng(100 + seed)
  nc, things = 5, [1, 2, 4]
  m = PanopticQuality(nc, things, 0, min_gt_points=6)
  scans = []
  for _ in range(4):
    n = 400
    gi = rng.integers(0, 9, n)
    gc = np.where(gi > 0, rng.choice(things, 9)[gi], rng.integers(0, nc, n))
    # predictions: the gt relabelled in blocks, so that some segments match, some split, some merge
    pi = np.where(rng.random(n) < 0.8, gi, rng.integers(0, 12, n))
    pi = np.where(rng.random(n) < 0.1, 0, pi)
    pc = np.where(rng.random(n) < 0.9, gc, rng.integers(0, nc, n))
    scans.append((gc, gi, pc, pi))
    m.update(gc, gi, pc, pi)
  tp, fp, fn, s = brute_force_pq([tuple(a.tolist() for a in sc) for sc in scans], set(things), 0, 6, nc)
  r = m.result()
  assert r["tp"].tolist() == tp[things].tolist() and r["fp"].tolist() == fp[things].tolist()
  assert r["fn"].tolist() == fn[things].tolist()
  assert np.allclose(r["pq"] * (tp + 0.5 * fp + 0.5 * fn)[things], s[things])
  assert tp.sum() > 0 and fp.sum() > 0 and fn.sum() > 0


# ---- argument checks of the C entry points (all before any CUDA call) ----

def call(B=2, Hh=64, Ww=512, nc=20, mask=0b10, ry=1, rx=2, wrap=1, tau=0.5, min_points=10, scratch=16, total=100,
         counts=16):
  lib = _lib.load()
  return lib.pcls_point_instances(None, 16, 16, B, Hh, Ww, total, None, None, None, nc, mask, ry, rx, wrap, tau,
                                  min_points, scratch, None, counts, None), lib.pcls_last_error().decode()


@pytest.mark.parametrize("kw,word", [
  (dict(ry=5), "ry"), (dict(ry=-1), "ry"), (dict(rx=9), "rx"), (dict(rx=-1), "rx"), (dict(ry=0, rx=0), "ry + rx"),
  (dict(wrap=2), "wrap"), (dict(Ww=4, rx=2), "2 rx < W"), (dict(tau=0.0), "tau"), (dict(tau=-1.0), "tau"),
  (dict(tau=float("nan")), "tau"), (dict(tau=float("inf")), "tau"), (dict(min_points=0), "min_points"),
  (dict(nc=33), "num_classes"), (dict(nc=0), "num_classes"), (dict(nc=4, mask=0b10000), "thing_mask"),
  (dict(B=70000, Hh=128, Ww=512), "2^31"), (dict(B=-1), "sizes"), (dict(total=-1), "sizes"),
  (dict(scratch=None), "NULL"), (dict(counts=None), "NULL"), (dict(scratch=8), "aligned"), (dict(), "NULL"),
])
def test_point_instances_argument_checks(kw, word):
  status, msg = call(**kw)
  assert status == -1
  assert msg.startswith("pcls_point_instances") and word in msg, msg


def test_point_instances_accepts_the_limits_before_its_buffers():
  # the window limits and wrap with 2 rx == W - 1 pass the parameter checks (the call then fails on NULL buffers)
  for kw in (dict(ry=4, rx=8), dict(ry=0, rx=1), dict(ry=1, rx=0), dict(Ww=5, rx=2), dict(Ww=4, rx=2, wrap=0),
             dict(nc=32, mask=0xFFFFFFFF), dict(tau=1e-30), dict(min_points=1)):
    status, msg = call(**kw)
    assert status == -1 and "NULL" in msg, (kw, msg)
  lib = _lib.load()
  assert lib.pcls_point_instances(None, None, 16, 0, 64, 512, 0, None, None, None, 20, 2, 1, 2, 1, 0.5, 10, None, None,
                                  None, None) == 0                   # B 0: nothing to do


def test_scratch_bytes():
  lib = _lib.load()
  assert lib.pcls_point_instances_scratch_bytes(64, 64, 2048) == 24 * 64 * 64 * 2048
  assert lib.pcls_point_instances_scratch_bytes(0, 64, 2048) == 0
  assert lib.pcls_point_instances_scratch_bytes(1, 0, 8) == -1
  assert lib.pcls_point_instances_scratch_bytes(1 << 14, 1 << 9, 1 << 8) == -1
  assert b"2^31" in lib.pcls_last_error()
