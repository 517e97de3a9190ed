"""Semantic map fusion on the GPU (pcls_semantic_map_*, SemanticMap, segment_scans --map): vote, growth, export and
query bit for bit against oracle/semantic_map.py on synthetic sequences with km-scale poses, a static scene whose fused
labels beat the per-scan ones, and the two-pass CLI on a tiny KITTI-layout sequence."""
import os

import numpy as np
import pytest
import torch

from oracle import semantic_map as SM
from tests.util import synth_scan

pytestmark = pytest.mark.gpu

NC, NONE = 20, 0
THINGS = tuple(range(1, 9))


def random_pose(rng, trans=5000.0, tilt_deg=4.0):
  """SE(3) with any yaw, a few degrees of roll and pitch and a translation up to +-trans metres."""
  yaw, roll, pitch = rng.uniform(-np.pi, np.pi), *np.deg2rad(rng.uniform(-tilt_deg, tilt_deg, 2))
  cz, sz, cx, sx, cy, sy = np.cos(yaw), np.sin(yaw), np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch)
  rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
  rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
  ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
  p = np.eye(4)
  p[:3, :3] = rz @ ry @ rx
  p[:3, 3] = rng.uniform(-trans, trans, 3) * np.array([1, 1, 0.01])
  return p


def sequence(seed, trans=5000.0):
  """12 scans near the origin of their own frame with poses spread over +-trans metres, labels that include "None" and
  ids outside [0, NC), and a few points with no voxel (NaN, and beyond 2^20 voxels).  Scans 6 .. 11 revisit scans 0 .. 5
  (the same points, new labels): 6 .. 8 from the same pose, so that voxels gather votes from several scans, 9 .. 11 from
  a pose moved by up to a metre."""
  rng = np.random.default_rng(seed)
  scans = []
  for i in range(6):
    s = synth_scan(rng, int(rng.integers(15000, 25000)))
    s[:5, 0] = np.nan
    s[5:8, 1] = 1e9
    scans.append(s)
  scans += [s.copy() for s in scans]
  labels = [rng.integers(-2, NC + 3, s.shape[0]).astype(np.int32) for s in scans]
  poses = [random_pose(rng, trans) for _ in range(6)]
  poses = np.stack(poses + poses[:3] + [p @ random_pose(rng, 1.0, 1.0) for p in poses[3:]])
  return scans, labels, poses


def batch(scans, lo, hi):
  sizes = [s.shape[0] for s in scans[lo:hi]]
  pts = torch.from_numpy(np.concatenate(scans[lo:hi])).cuda()
  offs = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).cuda()
  return pts, offs


def vote_all(m, scans, labels, poses, per_call):
  caps = []
  for lo in range(0, len(scans), per_call):
    pts, offs = batch(scans, lo, lo + per_call)
    m.vote(pts, offs, poses[lo:lo + per_call], torch.from_numpy(np.concatenate(labels[lo:lo + per_call])).cuda())
    caps.append(m.capacity)
  return caps


def oracle_table(scans, labels, poses, s, min_range=0.0, max_range=0.0, ignore=NONE):
  ks, ls = [], []
  for pts, lab, p in zip(scans, labels, poses):
    k, l = SM.voters(pts, [0, pts.shape[0]], p[None], s, lab, NC, ignore, min_range, max_range)
    ks.append(k)
    ls.append(l)
  return SM.table(np.concatenate(ks), np.concatenate(ls), NC)


def assert_export_equal(got, want):
  assert set(got) == {"voxels", "counts", "labels", "voxel_size"}
  for k in ("voxels", "counts", "labels"):
    assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), k
  assert float(got["voxel_size"]) == float(want["voxel_size"])


@pytest.mark.parametrize("voxel", [0.1, 0.25])
@pytest.mark.parametrize("limits", [(0.0, 0.0), (3.0, 50.0)])
def test_vote_and_export_equal_the_oracle(voxel, limits):
  from pclsegmentation_b200.semantic_map import SemanticMap
  scans, labels, poses = sequence(1)
  m = SemanticMap(NC, voxel_size=voxel, min_range=limits[0], max_range=limits[1], ignore_class=NONE)
  vote_all(m, scans, labels, poses, 4)
  keys, counts = oracle_table(scans, labels, poses, voxel, *limits)
  want = SM.export(keys, counts, voxel)
  assert (want["voxels"] < 0).any() and (want["voxels"] > 0).any()
  assert (counts.sum(1) > 1).sum() > 1000, "voxels should gather votes of several scans"
  assert m.num_voxels == len(keys)
  assert_export_equal(m.export(), want)


def test_boundary_points_fall_in_the_oracle_voxels():
  from pclsegmentation_b200.semantic_map import SemanticMap
  k = np.arange(-12, 13) * 0.25
  near = np.concatenate([k, np.nextafter(k, np.inf), np.nextafter(k, -np.inf), [-0.0, 0.0]]).astype(np.float32)
  g = np.stack(np.meshgrid(near, near[::7], near[::5], indexing="ij"), -1).reshape(-1, 3)
  pts = np.concatenate([g, np.zeros((g.shape[0], 1), np.float32)], 1)
  lab = (np.arange(pts.shape[0]) % 5).astype(np.int32)
  m = SemanticMap(5, voxel_size=0.25, max_range=0.0)
  pose = np.eye(4)[None]
  m.vote(pts, np.array([0, pts.shape[0]], np.int64), pose, lab)
  keys, counts = SM.table(*SM.voters(pts, [0, pts.shape[0]], pose, 0.25, lab, 5), 5)
  assert_export_equal(m.export(), SM.export(keys, counts, 0.25))
  assert SM.unpack_keys(SM.voxel_keys(np.float32([[-0.0, -0.25, 0.25, 0]]), [0, 1], pose, 0.25)[0]).tolist() == \
      [[0, -1, 1]]


def test_growth_keeps_the_map():
  from pclsegmentation_b200.semantic_map import SemanticMap
  scans, labels, poses = sequence(2)
  one = SemanticMap(NC, voxel_size=0.1, ignore_class=NONE, capacity=64)
  caps = vote_all(one, scans, labels, poses, 1)
  assert len(set(caps)) >= 3 and caps[0] > 64, caps        # grows from 64 at the first call and twice more
  assert 2 * one.num_voxels <= caps[-1]
  small = SemanticMap(NC, voxel_size=0.1, ignore_class=NONE, capacity=64)
  assert vote_all(small, scans, labels, poses, 2)[0] > 64
  big = SemanticMap(NC, voxel_size=0.1, ignore_class=NONE, capacity=1 << 22)
  vote_all(big, scans, labels, poses, 6)
  keys, counts = oracle_table(scans, labels, poses, 0.1, 0.0, 50.0)
  want = SM.export(keys, counts, 0.1)
  for m in (small, big, one):
    assert_export_equal(m.export(), want)


def test_query_equals_the_oracle_and_repeats():
  from pclsegmentation_b200.semantic_map import SemanticMap
  scans, labels, poses = sequence(3)
  vote_scans = 8          # scans 8 .. 11 never vote; they revisit the places scans 2 .. 5 voted
  keys, counts = oracle_table(scans[:vote_scans], labels[:vote_scans], poses[:vote_scans], 0.2, 0.0, 50.0)
  pts, offs = batch(scans, 0, len(scans))
  lab_all = np.concatenate(labels)
  thing_mask = sum(1 << c for c in THINGS)
  outs = []
  for run in range(2):
    m = SemanticMap(NC, voxel_size=0.2, ignore_class=NONE, capacity=1 << 10)
    vote_all(m, scans[:vote_scans], labels[:vote_scans], poses[:vote_scans], 3)
    for keep in ((), THINGS):
      for mv in (1, 3):
        got = m.relabel(pts, offs, poses, torch.from_numpy(lab_all).cuda(), keep_classes=keep, min_votes=mv)
        want = np.concatenate([SM.relabel(s, [0, s.shape[0]], p[None], 0.2, l, keys, counts,
                                          thing_mask if keep else 0, mv)
                               for s, l, p in zip(scans, labels, poses)])
        g = got.cpu().numpy()
        assert g.dtype == np.int32 and np.array_equal(g, want), (keep, mv)
        outs.append(g)
  assert (outs[0] != lab_all).sum() > 1000 and not np.array_equal(outs[0], outs[1])
  for a, b in zip(outs[:4], outs[4:]):
    assert np.array_equal(a, b)


def test_bad_poses_are_refused():
  from pclsegmentation_b200.semantic_map import SemanticMap
  m = SemanticMap(NC)
  pts = np.zeros((4, 4), np.float32)
  offs = np.array([0, 4], np.int64)
  lab = np.ones(4, np.int32)
  for bad in (np.eye(4)[None] * np.array([1, 1, 1, 2.0])[None, :, None], np.full((1, 4, 4), np.nan),
              np.eye(4, dtype=np.float32)[None], np.eye(4)[None].repeat(2, 0)):
    with pytest.raises(ValueError):
      m.vote(pts, offs, bad, lab)
  m.vote(pts, offs, torch.eye(4, dtype=torch.float64).cuda()[None], lab)
  assert m.num_voxels == 1


def static_scene(rng, n=40000):
  """World points on a ground plane and a few boxes, labelled by 2 m cells (so a 0.2 m voxel has one true class)."""
  g = np.stack([rng.uniform(-30, 30, n), rng.uniform(-30, 30, n), np.zeros(n)], 1)
  b = np.stack([rng.uniform(-30, 30, n // 2), rng.uniform(-30, 30, n // 2), rng.uniform(0.1, 3, n // 2)], 1)
  w = np.concatenate([g, b])
  cell = np.floor(w[:, :2] / 2.0).astype(np.int64)
  truth = (1 + (cell[:, 0] * 7 + cell[:, 1] * 3) % (NC - 1)).astype(np.int32)
  return w, truth


def test_fusion_beats_per_scan_labels_on_a_static_scene():
  from pclsegmentation_b200.semantic_map import SemanticMap
  rng = np.random.default_rng(5)
  world, truth = static_scene(rng)
  poses = np.stack([random_pose(rng, trans=5.0, tilt_deg=2.0) for _ in range(8)])
  scans, labels, truths = [], [], []
  for p in poses:
    idx = np.sort(rng.choice(world.shape[0], int(0.7 * world.shape[0]), replace=False))
    local = (np.linalg.inv(p) @ np.concatenate([world[idx], np.ones((idx.size, 1))], 1).T).T[:, :3]
    scans.append(np.concatenate([local, np.zeros((idx.size, 1))], 1).astype(np.float32))
    lab = truth[idx].copy()
    flip = rng.random(idx.size) < 0.2
    lab[flip] = rng.integers(1, NC, int(flip.sum()))
    labels.append(lab)
    truths.append(truth[idx])
  m = SemanticMap(NC, voxel_size=0.2, max_range=0.0, ignore_class=NONE)
  vote_all(m, scans, labels, poses, 4)
  pts, offs = batch(scans, 0, len(scans))
  lab_all, truth_all = np.concatenate(labels), np.concatenate(truths)
  fused = m.relabel(pts, offs, poses, torch.from_numpy(lab_all).cuda()).cpu().numpy()
  keys, counts = oracle_table(scans, labels, poses, 0.2)
  want = np.concatenate([SM.relabel(s, [0, s.shape[0]], p[None], 0.2, l, keys, counts)
                         for s, l, p in zip(scans, labels, poses)])
  assert np.array_equal(fused, want)
  per_scan, acc = (lab_all == truth_all).mean(), (fused == truth_all).mean()
  assert per_scan < 0.85 and acc > per_scan + 0.1, (per_scan, acc)


def _kitti_sequence(tmp_path, rng, n_scans=6):
  seq = tmp_path / "seq"
  (seq / "velodyne").mkdir(parents=True)
  (seq / "labels").mkdir()
  raw_of_class = np.array([0, 10, 11, 15, 18, 20, 30, 31, 32, 40, 44, 48, 49, 50, 51, 70, 71, 72, 80, 81], np.uint32)
  cams = []
  for i in range(n_scans):
    pts = synth_scan(rng, int(rng.integers(6000, 9000)))
    pts[:, :3] *= 0.15         # ranges 0.3 .. 12 m: voxels near the sensor hold several points of one scan
    pts.tofile(str(seq / "velodyne" / ("%06d.bin" % i)))
    raw_of_class[rng.integers(0, NC, pts.shape[0])].tofile(str(seq / "labels" / ("%06d.label" % i)))
    c = np.eye(4)
    c[:3, 3] = [0.1 * i, 0.02 * i, 1.5 * i]      # the camera frame's z is forward
    cams.append(c)
  (seq / "poses.txt").write_text("\n".join(" ".join("%.12e" % v for v in c[:3].reshape(-1)) for c in cams) + "\n")
  tr = "4.27e-04 -9.99967e-01 -8.08e-03 -1.198e-02 -7.21e-03 8.08e-03 -9.99941e-01 -5.404e-02 " \
       "9.99973e-01 4.85e-04 -7.21e-03 -2.921e-01"
  (seq / "calib.txt").write_text("P0: " + " ".join(["0"] * 12) + "\nTr: " + tr + "\n")
  return seq, raw_of_class


def test_segment_scans_map_cli(tmp_path, capsys):
  import yaml
  from pclsegmentation_b200 import segment_scans
  from pclsegmentation_b200.dataset_convert import learning_map_lut
  from pclsegmentation_b200.pipeline import Clustering
  from pclsegmentation_b200.semantic_map import kitti_lidar_poses
  from pclsegmentation_b200.utils.args_loader import load_model_config
  rng = np.random.default_rng(21)
  seq, raw_of_class = _kitti_sequence(tmp_path, rng)
  mc, model = load_model_config("squeezesegv2", "squeezesegv2kitti")
  model.randomize_batch_norm(1)
  wpath = str(tmp_path / "weights.npz")
  model.save_weights_npz(wpath)
  learning_map = {int(r): c for c, r in enumerate(raw_of_class)}
  ypath = tmp_path / "map.yaml"
  ypath.write_text(yaml.safe_dump({"learning_map": learning_map,
                                   "learning_map_inv": {c: int(r) for c, r in enumerate(raw_of_class)}}))
  base = ["--scans", str(seq / "velodyne" / "*.bin"), "-m", "squeezesegv2", "-n", "squeezesegv2kitti", "-p", wpath,
          "--batch", "2", "--learning_map", str(ypath)]
  mapped = ["--map", "--poses", str(seq / "poses.txt"), "--calib", str(seq / "calib.txt")]
  segment_scans.main(base + ["--output_dir", str(tmp_path / "plain")])
  capsys.readouterr()
  rep = segment_scans.main(base + mapped + ["--map_out", str(tmp_path / "map.npz"), "--output_dir",
                                            str(tmp_path / "fused"), "--labels", str(seq / "labels" / "*.label")])
  printed = capsys.readouterr().out
  assert "FUSED (semantic map)" in printed and printed.count("MIoU:") == 2
  assert "fused" in rep and 0.0 <= rep["fused"]["miou"] <= 1.0
  lut = learning_map_lut(learning_map)
  poses = kitti_lidar_poses(str(seq / "poses.txt"), str(seq / "calib.txt"))
  files = sorted(os.listdir(str(seq / "velodyne")))
  scans = [np.fromfile(str(seq / "velodyne" / f), np.float32).reshape(-1, 4) for f in files]
  first = [lut[np.fromfile(str(tmp_path / "plain" / f.replace(".bin", ".label")), np.uint32)].astype(np.int32)
           for f in files]
  keys, counts = oracle_table(scans, first, poses, 0.2, 0.0, 50.0, mc.CLASSES.index("None"))
  with np.load(str(tmp_path / "map.npz")) as f:
    assert_export_equal({k: f[k] for k in f.files}, SM.export(keys, counts, 0.2))
  thing_mask = Clustering().thing_mask(mc)
  changed = 0
  for f, s, l, p in zip(files, scans, first, poses):
    want = SM.relabel(s, [0, s.shape[0]], p[None], 0.2, l, keys, counts, thing_mask, 1)
    got = np.fromfile(str(tmp_path / "fused" / f.replace(".bin", ".label")), np.uint32)
    assert np.array_equal(got, raw_of_class[want])
    changed += int((want != l).sum())
  assert changed > 0
  # refused combinations
  out = ["--output_dir", str(tmp_path / "refused")]
  for extra, msg in ((["--instances"], "cannot be combined"), (["--confidence"], "cannot be combined"),
                     (["--mc_dropout", "2"], "cannot be combined"), (["--format", "nuscenes"], "no nuScenes poses"),
                     ([], "needs --poses")):
    args = base + out + (mapped if msg != "needs --poses" else ["--map"]) + extra
    with pytest.raises(SystemExit, match=msg):
      segment_scans.main(args)
  odd = tmp_path / "odd"
  odd.mkdir()
  scans[0].tofile(str(odd / "first.bin"))
  with pytest.raises(SystemExit, match="not a scan number"):
    segment_scans.main(["--scans", str(odd / "*.bin")] + base[2:] + mapped + out)
