"""Dataset statistics, host side: the oracle on a hand-computed frame, the order-free combination of per-frame rows, the
CLI's argument parsing and JSON keys, and the two-rank gather (gloo) - all without a GPU."""
import json
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import dataset_stats as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200 import dataset_stats as DS

nan, inf = float("nan"), float("inf")


def test_oracle_hand_computed_2x3_frame():
  # (x, y, z, remission, range, label); valid = range > 0
  f = np.array([[[1.0, 2.0, 3.0, 0.5, 10.0, 2.7],       # valid, label 2 (truncated)
                 [nan, nan, nan, nan, 0.0, nan],         # invalid: range 0, NaN elsewhere is ignored
                 [3.0, -2.0, 1.0, 0.25, 20.0, -0.5]],    # valid, label -0.5 truncates to 0
                [[9.0, 9.0, 9.0, 9.0, -1.0, 1.0],        # invalid: negative range
                 [5.0, 0.0, -1.0, 0.75, 30.0, 7.0],      # valid, label 7 not in [0, 3): dropped
                 [0.0, 0.0, 0.0, 0.0, nan, 1.0]]])       # invalid: NaN range
  s = np.array([1.0, 0.0, 0.0, 0.0, 0.0])
  o = O.frame_stats(f[None], s, num_classes=3)
  assert o["frame_valid"].tolist() == [3]
  assert o["row_valid"].tolist() == [2, 1] and o["col_valid"].tolist() == [1, 1, 1]
  fs = o["frame_sums"][0]
  # x: values 1, 3, 5, d = 0, 2, 4
  assert fs[0].tolist() == [6.0, 20.0, 1.0, 5.0]
  assert fs[1].tolist() == [0.0, 8.0, -2.0, 2.0]
  assert fs[2].tolist() == [3.0, 11.0, -1.0, 3.0]
  assert fs[3].tolist() == [1.5, 0.25 + 0.0625 + 0.5625, 0.25, 0.75]
  assert fs[4].tolist() == [60.0, 1400.0, 10.0, 30.0]
  assert o["class_pixels"].tolist() == [1, 0, 1] and o["dropped"] == 1
  # NaN labels at valid pixels and non-finite values are dropped; NaN values stay out of min / max
  g = f.copy()
  g[0, 0, 5], g[0, 2, 5], g[0, 0, 1] = nan, inf, nan
  o = O.frame_stats(g[None], None, num_classes=3)
  assert o["class_pixels"].tolist() == [0, 0, 0] and o["dropped"] == 3
  assert math.isnan(o["frame_sums"][0, 1, 0]) and o["frame_sums"][0, 1, 2:].tolist() == [-2.0, 0.0]
  # a frame with no valid pixel
  e = O.frame_stats(np.zeros((1, 2, 3, 5)))
  assert e["frame_sums"][0, :, :2].tolist() == [[0.0, 0.0]] * 5
  assert (e["frame_sums"][0, :, 2] == inf).all() and (e["frame_sums"][0, :, 3] == -inf).all()


def _synthetic_state(rng, F, H=4, W=8, nc=5):
  sums = np.empty((F, 5, 4))
  sums[:, :, 0] = rng.normal(0, 1e3, (F, 5))
  sums[:, :, 1] = rng.uniform(1e6, 1e8, (F, 5))
  sums[:, :, 2] = rng.normal(-50, 5, (F, 5))
  sums[:, :, 3] = rng.normal(50, 5, (F, 5))
  return dict(frame_sums=sums, frame_valid=rng.integers(1000, 5000, F), row_valid=rng.integers(0, 100, H),
              col_valid=rng.integers(0, 100, W), class_pixels=rng.integers(0, 1000, nc), dropped=3)


def test_combine_is_order_free_and_matches_the_closed_form():
  rng = np.random.default_rng(0)
  st = _synthetic_state(rng, 200)
  shift = np.array([1.0, -2.0, 0.5, 0.25, 8.0])
  ref = DS.combine(st, shift, 4, 8)
  for seed in range(5):
    p = np.random.default_rng(seed).permutation(200)
    perm = dict(st, frame_sums=st["frame_sums"][p], frame_valid=st["frame_valid"][p])
    got = DS.combine(perm, shift, 4, 8)
    for k in ("mean", "std", "min", "max"):
      assert got[k].tobytes() == ref[k].tobytes(), k
  # the float64 closed form, with exact sums
  n = int(st["frame_valid"].sum())
  for c in range(5):
    m1 = math.fsum(st["frame_sums"][:, c, 0]) / n
    m2 = math.fsum(st["frame_sums"][:, c, 1]) / n
    assert ref["mean"][0, 0, c] == shift[c] + m1
    assert ref["std"][0, 0, c] == math.sqrt(max(m2 - m1 * m1, 0.0))
  assert ref["mean"].shape == ref["std"].shape == (1, 1, 5) and ref["mean"].dtype == np.float64
  assert ref["frames"] == 200 and ref["pixels"] == 200 * 32 and ref["valid"] == n
  assert np.array_equal(ref["min"], st["frame_sums"][:, :, 2].min(0))
  assert np.array_equal(ref["row_valid_fraction"], st["row_valid"] / (200 * 8))
  assert np.array_equal(ref["col_valid_fraction"], st["col_valid"] / (200 * 4))
  assert np.isclose(ref["class_frequency"].sum(), 1.0)
  # no valid pixel at all: NaN moments, not an exception
  empty = DS.combine(dict(st, frame_valid=np.zeros(200, np.int64)), shift, 4, 8)
  assert np.isnan(empty["mean"]).all() and np.isnan(empty["std"]).all()


def test_cli_parses_both_modes_and_json_has_the_documented_keys(tmp_path):
  ap = DS.build_parser()
  a = ap.parse_args(["-d", "out/train/*.npy", "-n", "squeezesegv2kitti", "-b", "16", "--json", "s.json"])
  assert (a.data, a.scans, a.config, a.batch, a.json, a.no_labels) == \
      ("out/train/*.npy", None, "squeezesegv2kitti", 16, "s.json", False)
  assert ap.parse_args(["-d", "x/*.npy", "--no_labels"]).no_labels
  a = ap.parse_args(["--scans", "seq/*/velodyne/*.bin", "--format", "nuscenes", "--width", "2048", "--labels", "l/*",
                     "--learning_map", "m.yaml", "--ring", "-n", "squeezesegv2nuscenes"])
  assert (a.scans, a.format, a.width, a.height, a.fov_up, a.fov_down, a.ring, a.batch) == \
      ("seq/*/velodyne/*.bin", "nuscenes", 2048, None, None, None, True, 64)
  rep = DS.combine(_synthetic_state(np.random.default_rng(1), 10), np.zeros(5), 4, 8)
  assert set(rep) == set(DS.KEYS)
  p = tmp_path / "s.json"
  p.write_text(json.dumps(DS.to_json(rep)))
  back = json.loads(p.read_text())
  assert set(back) == set(DS.KEYS) and len(back["mean"][0][0]) == 5 and len(back["row_valid_fraction"]) == 4
  # the report prints the config lines and the check against the config
  from pclsegmentation_b200.utils.args_loader import config_map
  mc = config_map["squeezesegv2kitti"]()
  dm, ds = DS.config_check(dict(rep, mean=mc.INPUT_MEAN.copy(), std=mc.INPUT_STD.copy()), mc)
  assert np.allclose(dm, 0) and np.allclose(ds, 1)


def test_c_argument_checks_without_gpu():
  lib = _lib.load()
  args = lambda **kw: [kw.get("frames"), kw.get("dtype", 1), kw.get("channels", 6), kw.get("B", 1), kw.get("H", 4),
                       kw.get("W", 8),
                       None, kw.get("nc", 20), None, None, None, None, kw.get("cls"), None, None]
  assert lib.pcls_dataset_stats(*args(dtype=2)) == -1 and b"dtype" in lib.pcls_last_error()
  assert lib.pcls_dataset_stats(*args(channels=4)) == -1 and b"channels" in lib.pcls_last_error()
  assert lib.pcls_dataset_stats(*args(W=16385)) == -1
  assert lib.pcls_dataset_stats(*args(H=16385)) == -1 and b"H <= 16384" in lib.pcls_last_error()
  assert lib.pcls_dataset_stats(*args(nc=33, cls=8)) == -1 and b"num_classes" in lib.pcls_last_error()
  assert lib.pcls_dataset_stats(*args(channels=5, cls=8)) == -1
  assert lib.pcls_dataset_stats(*args()) == -1 and b"NULL" in lib.pcls_last_error()
  assert lib.pcls_dataset_stats(*args(B=0)) == 0


def _free_port():
  with socket.socket() as s:
    s.bind(("127.0.0.1", 0))
    return s.getsockname()[1]


def _worker(rank, world, port, states, out):
  os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
  dist.init_process_group("gloo", rank=rank, world_size=world)
  try:
    from pclsegmentation_b200.sharding import Communicator
    st = DS.DatasetStats(5, 4, 8, shift=np.arange(5.0))
    st.state = lambda: states[rank]                        # this rank's device rows, as update() leaves them
    rep = st.finish(Communicator())
    out[rank] = {k: (v.tobytes() if isinstance(v, np.ndarray) else v) for k, v in rep.items()}
  finally:
    dist.destroy_process_group()


def test_two_rank_finish_equals_single_rank_bit_for_bit():
  rng = np.random.default_rng(7)
  full = _synthetic_state(rng, 13)
  states = []
  for lo, hi in ((0, 7), (7, 13)):
    states.append(dict(frame_sums=full["frame_sums"][lo:hi], frame_valid=full["frame_valid"][lo:hi],
                       row_valid=rng.integers(0, 50, 4), col_valid=rng.integers(0, 50, 8),
                       class_pixels=rng.integers(0, 500, 5), dropped=int(rng.integers(0, 9))))
  full = dict(full, row_valid=states[0]["row_valid"] + states[1]["row_valid"],
              col_valid=states[0]["col_valid"] + states[1]["col_valid"],
              class_pixels=states[0]["class_pixels"] + states[1]["class_pixels"],
              dropped=states[0]["dropped"] + states[1]["dropped"])
  mgr = mp.Manager()
  out = mgr.dict()
  mp.spawn(_worker, args=(2, _free_port(), states, out), nprocs=2, join=True)
  solo = DS.DatasetStats(5, 4, 8, shift=np.arange(5.0))
  solo.state = lambda: full
  ref = {k: (v.tobytes() if isinstance(v, np.ndarray) else v) for k, v in solo.finish().items()}
  assert out[0] == ref and out[1] == ref
