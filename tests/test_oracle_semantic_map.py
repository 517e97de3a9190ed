"""Semantic map fusion (pcls_semantic_map_*): hand-built cases that pin each rule of the contract on the numpy oracle,
the KITTI pose composition, the scan-to-pose and growth rules of the Python layer, and the argument checks of the C
entry points, which run before any CUDA call (no GPU needed)."""
import numpy as np
import pytest

from oracle import semantic_map as SM
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.semantic_map import grown_capacity, kitti_lidar_poses, scan_pose_index, unpack_keys

EYE = np.eye(4)[None]


def keys_of(xyz, s=0.25, pose=EYE):
  pts = np.concatenate([np.asarray(xyz, np.float32).reshape(-1, 3), np.zeros((len(xyz), 1), np.float32)], 1)
  return SM.voxel_keys(pts, [0, len(pts)], pose, s)


def test_key_packing_and_floor_of_negative_and_boundary_coordinates():
  k, ok = keys_of([[0.0, 0.0, 0.0], [-0.0, 0.25, -0.25], [0.24, -0.01, 0.5], [-0.26, 1.0, -1.0]])
  assert ok.all()
  want = [(0, 0, 0), (0, 1, -1), (0, -1, 2), (-2, 4, -4)]
  assert [int(v) for v in k] == [int(SM.pack_key(*v)) for v in want]
  assert unpack_keys(k).tolist() == [list(v) for v in want] == SM.unpack_keys(k).tolist()
  assert int(SM.pack_key(0, 0, 0)) == (1 << 62) | (1 << 41) | (1 << 20)
  assert int(SM.pack_key(2 ** 20 - 1, 2 ** 20 - 1, 2 ** 20 - 1)) == (1 << 63) - 1      # always below 2^63
  assert int(SM.pack_key(-2 ** 20, -2 ** 20, -2 ** 20)) == 0


def test_world_coordinates_are_rounded_product_by_product():
  # a rotation and a km-scale translation: the key comes from ((r0 x + r1 y) + r2 z) + t in float64, no FMA
  pose = np.eye(4)
  pose[:3, :3] = [[0.6, -0.8, 0.0], [0.8, 0.6, 0.0], [0.0, 0.0, 1.0]]
  pose[:3, 3] = [-4321.123, 987.5, 3.3]
  p = np.float32([1.1, -7.3, 0.7])
  x, y, z = (np.float64(v) for v in p)
  wx = ((0.6 * x + -0.8 * y) + 0.0 * z) + -4321.123
  k, ok = keys_of([p], s=0.1, pose=pose[None])
  assert ok[0] and SM.unpack_keys(k)[0, 0] == np.floor(wx / 0.1)


def test_points_without_a_voxel():
  big = 0.25 * 2 ** 20
  k, ok = keys_of([[np.nan, 0, 0], [0, np.inf, 0], [big, 0, 0], [-big, 0, 0], [0, 0, -big - 0.25],
                   [big - 0.25, 0, 0]])
  assert ok.tolist() == [False, False, False, True, False, True]
  assert unpack_keys(k[ok]).tolist() == [[-2 ** 20, 0, 0], [2 ** 20 - 1, 0, 0]]
  # a non-finite pose entry makes every point of its scan voxel-less
  pose = np.eye(4)[None].copy()
  pose[0, 1, 3] = np.inf
  assert not keys_of([[1, 1, 1]], pose=pose)[1].any()


def vote_table(xyz, labels, nc=4, **kw):
  pts = np.concatenate([np.asarray(xyz, np.float32).reshape(-1, 3), np.zeros((len(xyz), 1), np.float32)], 1)
  vk, vl = SM.voters(pts, [0, len(pts)], EYE, 1.0, labels, nc, **kw)
  return pts, SM.table(vk, vl, nc)


def test_argmax_ties_to_the_lowest_class_and_vote_filters():
  xyz = [[0.5, 0.5, 0.5]] * 6 + [[5.5, 0.5, 0.5]] * 3
  labels = [2, 1, 2, 1, 9, -1, 3, 3, 0]            # 9 and -1 are not classes and cast no vote
  pts, (keys, counts) = vote_table(xyz, labels)
  assert counts.tolist() == [[0, 2, 2, 0], [1, 0, 0, 2]]
  ex = SM.export(keys, counts, 1.0)
  assert ex["labels"].tolist() == [1, 3] and ex["voxels"].tolist() == [[0, 0, 0], [5, 0, 0]]
  _, (_, c_ign) = vote_table(xyz, labels, ignore_class=3)
  assert c_ign.tolist() == [[0, 2, 2, 0], [1, 0, 0, 0]]


def test_range_limits_apply_to_votes_in_the_sensor_frame():
  xyz = [[1.0, 0, 0], [3.0, 0, 0], [4.0, 0, 0], [0, 0, 5.0]]
  _, (keys, _) = vote_table(xyz, [1, 1, 1, 1], min_range=3.0, max_range=4.0)
  assert SM.unpack_keys(keys).tolist() == [[3, 0, 0], [4, 0, 0]]              # both limits inclusive
  _, (keys, _) = vote_table(xyz, [1, 1, 1, 1], min_range=3.0, max_range=0.0)  # max <= 0: no upper limit
  assert len(keys) == 3


def test_relabel_keep_mask_min_votes_and_unmapped_points():
  xyz = [[0.5, 0.5, 0.5]] * 3 + [[2.5, 0.5, 0.5]]
  pts, (keys, counts) = vote_table(xyz, [2, 2, 1, 3])
  q = np.concatenate([pts, np.float32([[9.5, 0, 0, 0], [np.nan, 0, 0, 0]])])
  lab = np.array([0, 1, 2, 0, 1, 1], np.int32)
  off = [0, len(q)]
  assert SM.relabel(q, off, EYE, 1.0, lab, keys, counts).tolist() == [2, 2, 2, 3, 1, 1]
  assert SM.relabel(q, off, EYE, 1.0, lab, keys, counts, keep_mask=0b10).tolist() == [2, 1, 2, 3, 1, 1]
  assert SM.relabel(q, off, EYE, 1.0, lab, keys, counts, min_votes=2).tolist() == [2, 2, 2, 0, 1, 1]
  assert SM.relabel(q, off, EYE, 1.0, lab, keys, counts, min_votes=4).tolist() == lab.tolist()


def _write(path, text):
  path.write_text(text)
  return str(path)


def test_kitti_lidar_poses(tmp_path):
  rng = np.random.default_rng(0)
  tr = np.eye(4)
  a = 0.3
  tr[:3, :3] = [[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]]
  tr[:3, 3] = [0.27, -0.08, -0.01]
  cams = np.tile(np.eye(4), (3, 1, 1))
  for i in range(3):
    b = rng.uniform(-np.pi, np.pi)
    cams[i, :3, :3] = [[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]]
    cams[i, :3, 3] = rng.uniform(-100, 100, 3)
  poses = _write(tmp_path / "poses.txt", "\n".join(" ".join("%.17g" % v for v in c[:3].reshape(-1)) for c in cams))
  calib = _write(tmp_path / "calib.txt", "P0: " + " ".join(["0"] * 12) + "\nTr: " +
                 " ".join("%.17g" % v for v in tr[:3].reshape(-1)) + "\n")
  got = kitti_lidar_poses(poses, calib)
  assert got.shape == (3, 4, 4) and got.dtype == np.float64
  want = np.stack([np.linalg.inv(tr) @ c @ tr for c in cams])
  assert np.allclose(got, want, rtol=0, atol=1e-12)
  # a lidar point p seen at pose i: world = inv(Tr) @ cam_i @ Tr @ p
  p = np.array([3.0, -2.0, 1.0, 1.0])
  assert np.allclose(got[1] @ p, np.linalg.inv(tr) @ (cams[1] @ (tr @ p)), atol=1e-9)
  ident = _write(tmp_path / "ident.txt", "Tr: 1 0 0 0 0 1 0 0 0 0 1 0\n")
  assert np.array_equal(kitti_lidar_poses(poses, ident), cams)
  with pytest.raises(ValueError):
    kitti_lidar_poses(poses, _write(tmp_path / "no_tr.txt", "P0: " + " ".join(["0"] * 12) + "\n"))


def test_scan_stem_gives_the_pose():
  assert scan_pose_index("/data/seq/08/velodyne/000123.bin", 200) == 123
  assert scan_pose_index("000000.bin", 1) == 0
  for bad in ("scan_a.bin", "12a.bin", "-1.bin"):
    with pytest.raises(ValueError):
      scan_pose_index(bad, 200)
  with pytest.raises(ValueError):
    scan_pose_index("000200.bin", 200)


def test_growth_rule_arithmetic():
  assert grown_capacity(64, 0, 32) == 64                    # load exactly 1/2: no growth
  assert grown_capacity(64, 0, 33) == 128
  assert grown_capacity(64, 10, 100) == 256                 # smallest power of two >= 220
  assert grown_capacity(1 << 20, 1000, 5000) == 1 << 20
  assert grown_capacity(1 << 10, 3000, 1096) == 8192        # 2 * 4096 exactly
  for cap, fill, n in ((64, 7, 500), (1024, 900, 1), (1 << 20, 300000, 250000)):
    c = grown_capacity(cap, fill, n)
    assert c & (c - 1) == 0 and 2 * (fill + n) <= c and (c == cap or c < 4 * (fill + n))


def test_c_abi_argument_checks_without_gpu():
  lib = _lib.load()
  P = 16                     # any non-NULL aligned address: the calls return before touching memory
  vote = lambda **kw: lib.pcls_semantic_map_vote(*[kw.get(n, d) for n, d in (
      ("points", P), ("offsets", P), ("B", 1), ("total", 10), ("poses", P), ("s", 0.2), ("lo", 0.0), ("hi", 50.0),
      ("labels", P), ("nc", 20), ("ignore", 0), ("keys", P), ("counts", P), ("cap", 64), ("state", P), ("st", None))])
  for kw, msg in (({"nc": 0}, b"num_classes"), ({"nc": 33}, b"num_classes"), ({"ignore": 20}, b"ignore_class"),
                  ({"ignore": -2}, b"ignore_class"), ({"s": 0.0}, b"voxel_size"), ({"s": float("nan")}, b"voxel_size"),
                  ({"lo": -1.0}, b"range"), ({"hi": 1.0, "lo": 2.0}, b"range"), ({"hi": float("inf")}, b"range"),
                  ({"cap": 48}, b"power of two"), ({"cap": 0}, b"power of two"), ({"total": 1 << 31}, b"2^31"),
                  ({"keys": None}, b"NULL"), ({"state": None}, b"NULL"), ({"poses": None}, b"NULL"),
                  ({"labels": None}, b"NULL"), ({"points": 8}, b"aligned")):
    assert vote(**kw) == -1, kw
    assert msg in lib.pcls_last_error(), (kw, lib.pcls_last_error())
  query = lambda **kw: lib.pcls_semantic_map_query(*[kw.get(n, d) for n, d in (
      ("points", P), ("offsets", P), ("B", 1), ("total", 10), ("poses", P), ("s", 0.2), ("labels", P), ("nc", 20),
      ("keep", 0), ("min_votes", 1), ("keys", P), ("counts", P), ("cap", 64), ("out", P), ("st", None))])
  for kw, msg in (({"keep": 1 << 20}, b"keep_mask"), ({"min_votes": 0}, b"min_votes"), ({"cap": 100}, b"power of two"),
                  ({"out": None}, b"NULL"), ({"nc": 40}, b"num_classes"), ({"s": -1.0}, b"voxel_size")):
    assert query(**kw) == -1, kw
    assert msg in lib.pcls_last_error(), (kw, lib.pcls_last_error())
  assert lib.pcls_semantic_map_grow(P, P, 64, 20, 32, 32, 96, P, None) == -1
  assert b"power" in lib.pcls_last_error()
  assert lib.pcls_semantic_map_grow(P, P, 64, 20, P, 32, 128, P, None) == -1
  assert b"must not be the old one" in lib.pcls_last_error()
  assert lib.pcls_semantic_map_grow(P, P, 64, 0, 32, 48, 128, P, None) == -1
  # nothing to do: returns before any launch, so it succeeds without a device
  assert vote(total=0) == 0 and query(total=0) == 0
