"""Per-point labels (pcls_point_labels): hand-built cases that pin each rule of the contract on the numpy oracle, and the
argument checks of the C entry points, which run before any CUDA call (no GPU needed)."""
import ctypes

import numpy as np
import pytest

from oracle import point_labels as PL
from pclsegmentation_b200 import _lib

NC, NONE = 5, 0


def grid(H=5, W=5, pred=1, rng_val=10.0):
  return np.full((H, W), pred, np.int32), np.full((H, W), rng_val, np.float32), np.ones((H, W), bool)


def one(pred, rng, valid, x, y, rho, **kw):
  return int(PL.point_labels(pred, rng, valid, [x], [y], [rho], NC, NONE, **kw)[0])


def test_search_1_is_the_pixel_label_and_dropped_points_get_none():
  pred, rng, valid = grid(pred=3)
  pred[2, 4] = 2
  out = PL.point_labels(pred, rng, valid, [4, -1, 0], [2, -1, 0], [10.0, 0.0, 5.0], NC, 4)
  assert out.tolist() == [2, 4, 3]          # none_index 4 for the dropped point, not 0


def test_distance_tie_goes_to_the_lower_entry():
  # 3x3 window around (2,2), k 2: the centre (d 0) and one neighbour at d 1 - entries j 1 (above) and 7 (below) tie
  pred, rng, valid = grid(pred=4, rng_val=50.0)
  pred[1, 2], rng[1, 2] = 1, 11.0           # j 1
  pred[3, 2], rng[3, 2] = 2, 9.0            # j 7, same |d| = 1
  pred[2, 2] = 3
  # votes: centre 3, j1 1 -> tie 1 vs 1 -> lowest class 1; had j 7 been taken it would be 2 (class 2 < 3)
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=2) == 1
  pred[1, 2], pred[3, 2] = 2, 1             # swap labels: j 1 (now class 2) still wins the tie on distance
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=2) == 2


def test_vote_tie_goes_to_the_lowest_class():
  pred, rng, valid = grid(pred=4, rng_val=50.0)
  pred[2, 2] = 3
  pred[2, 1], rng[2, 1] = 2, 10.0           # d 0
  pred[2, 3], rng[2, 3] = 2, 10.0
  pred[1, 2], rng[1, 2] = 3, 10.0
  # k 4: centre 3, (1,2) 3, (2,1) 2, (2,3) 2 -> 2 votes each -> class 2
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=4) == 2


def test_cutoff_at_equality_votes():
  pred, rng, valid = grid(pred=4, rng_val=50.0)
  pred[2, 2] = 3
  pred[2, 1], rng[2, 1] = 1, 10.5
  pred[2, 3], rng[2, 3] = 1, 9.5
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=3, cutoff=0.5) == 1    # d == cutoff votes: 1 wins 2:1
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=3, cutoff=0.49) == 3   # only the centre votes
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=3, cutoff=0.0) == 1    # no cutoff


def test_image_edges_are_invalid_without_wrap_around():
  pred, rng, valid = grid(H=3, W=6, pred=4, rng_val=50.0)
  pred[1, 0] = 3
  pred[:, 5], rng[:, 5] = 1, 10.0           # the last column: neighbours at d 0 only with column wrap-around
  # point at column 0, k 3: the centre (3) and the first two entries at d 40 - (0,0) and (0,1), both 4
  assert one(pred, rng, valid, 0, 1, 10.0, search=3, k=3) == 4
  # the same at row 0: window rows -1 (outside) .. 1
  pred[0, 0] = 3
  assert one(pred, rng, valid, 0, 0, 10.0, search=3, k=3) == 3   # centre 3, then (0,1) 4 and (1,0) 3
  # a neighbour in the previous row's last column must never be read for column 0
  pred2, rng2, valid2 = grid(H=3, W=4, pred=4, rng_val=50.0)
  valid2[:, :] = False
  valid2[1, 0] = True
  pred2[1, 0] = 2
  valid2[0, 3], pred2[0, 3], rng2[0, 3] = True, 1, 10.0
  assert one(pred2, rng2, valid2, 0, 1, 10.0, search=3, k=9) == 2


def test_centre_uses_the_point_range_and_the_pixel_label():
  # the point lost its pixel to a much nearer point (winner range 2): with the winner's range the centre would be far
  pred, rng, valid = grid(pred=4, rng_val=40.0)
  pred[2, 2], rng[2, 2] = 1, 2.0
  pred[2, 1], rng[2, 1] = 3, 30.5
  # k 1: the centre, d 0 with the point's own range 30 -> label 1 (pixel label); with the winner's range (d 28) the
  # nearest entry would be (2,1) at d 0.5 -> 3
  assert one(pred, rng, valid, 2, 2, 30.0, search=3, k=1) == 1
  # k 2, cutoff 1: the centre (1) and (2,1) (3) vote -> tie -> 1; the 4s at d 10 are not selected
  assert one(pred, rng, valid, 2, 2, 30.0, search=3, k=2, cutoff=1.0) == 1
  pred[2, 2] = 4
  assert one(pred, rng, valid, 2, 2, 30.0, search=3, k=2, cutoff=1.0) == 3


def test_ignore_class_and_the_fallback_when_nothing_votes():
  pred, rng, valid = grid(pred=0, rng_val=10.0)
  pred[2, 2] = 0
  pred[2, 1] = 2
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=9) == 0
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=9, ignore_class=0) == 2
  pred[2, 1] = 0
  # everything is class 0 and ignored: no votes -> the centre pixel's prediction
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=9, ignore_class=0) == 0
  pred[2, 2] = 3
  pred[:, :2] = 0
  rng[:, 3:] = 99.0
  pred[:, 3:] = 1
  # cutoff excludes the 1s, the 0s are ignored, the centre (3) votes
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=9, cutoff=1.0, ignore_class=0) == 3
  pred[2, 2] = 0
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=9, cutoff=1.0, ignore_class=0) == 0


def test_fewer_valid_entries_than_k():
  pred, rng, valid = grid(pred=2, rng_val=10.0)
  valid[:, :] = False
  valid[2, 2] = True
  pred[2, 2] = 1
  valid[1, 1], pred[1, 1], rng[1, 1] = True, 3, 10.0
  valid[3, 3], pred[3, 3], rng[3, 3] = True, 3, 10.2
  assert one(pred, rng, valid, 2, 2, 10.0, search=5, k=25) == 3   # all three valid entries vote: 3 twice


def test_weights_scale_the_distance():
  pred, rng, valid = grid(pred=4, rng_val=50.0)
  pred[2, 2] = 1
  pred[2, 1], rng[2, 1] = 2, 10.0 + 0.8
  pred[1, 2], rng[1, 2] = 3, 10.0 + 0.5
  w = np.ones(9, np.float32)
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=2, weights=w) == 1     # {1, 3}: tie -> 1
  w[1] = 4.0                                                                  # j 1 = (1,2): d 2.0 > 0.8
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=3, weights=w, cutoff=1.0) == 1
  pred[2, 2] = 4
  assert one(pred, rng, valid, 2, 2, 10.0, search=3, k=2, weights=w) == 2     # {4, 2} -> 2


def test_knn_weights_match_the_oracle():
  from pclsegmentation_b200.pipeline import KNN
  for s, sigma in ((3, 1.0), (5, 1.0), (5, 2.0), (9, 0.7)):
    w = KNN(search=s, sigma=sigma).weights()
    assert w.dtype == np.float32 and w.shape == (s * s,)
    assert np.array_equal(w, PL.window_weights(s, sigma))
    assert w[(s * s) // 2] == w.min() and (w >= 0).all()


def test_knn_defaults_resolve_none():
  from pclsegmentation_b200.pipeline import KNN
  from pclsegmentation_b200.utils.args_loader import config_map
  k = KNN()
  assert (k.search, k.k, k.sigma, k.cutoff) == (5, 5, 1.0, 1.0)
  assert k.ignore_index(config_map["darknet53kitti"]()) == 0
  assert k.ignore_index(config_map["squeezesegv2"]()) == config_map["squeezesegv2"]().CLASSES.index("None")
  assert KNN(ignore_class=-1).ignore_index(config_map["darknet53kitti"]()) == -1


# ---- argument checks of the C entry points (all before any CUDA call) ----

def call(search=5, k=5, num_classes=20, none_index=0, ignore_class=0, scratch=None, weights=None, cutoff=1.0):
  lib = _lib.load()
  w = None
  if weights is not None:
    w = (ctypes.c_float * len(weights))(*weights)
  return lib.pcls_point_labels(None, None, None, 2, 64, 512, 100, None, None, None, num_classes, none_index, search, k,
                               w, cutoff, ignore_class, scratch, None, None), lib.pcls_last_error().decode()


@pytest.mark.parametrize("kw,word", [
  (dict(search=4), "search"), (dict(search=0), "search"), (dict(search=11), "search"), (dict(search=-1), "search"),
  (dict(k=0), "k "), (dict(search=3, k=10), "k "), (dict(search=7, k=33), "k "),
  (dict(num_classes=33), "num_classes"), (dict(num_classes=0), "num_classes"),
  (dict(none_index=20), "none_index"), (dict(none_index=-1), "none_index"),
  (dict(ignore_class=20), "ignore_class"), (dict(ignore_class=-2), "ignore_class"),
  (dict(scratch=None), "pixel_scratch"),
  (dict(scratch=16, weights=[1.0] * 12 + [-1.0] + [1.0] * 12), "h_window_weights"),
  (dict(scratch=16, weights=[1.0] * 12 + [float("inf")] + [1.0] * 12), "h_window_weights"),
  (dict(scratch=16, cutoff=float("nan")), "cutoff"),
])
def test_point_labels_argument_checks(kw, word):
  status, msg = call(**kw)
  assert status == -1
  assert msg.startswith("pcls_point_labels") and word in msg, msg


def test_point_labels_null_buffers_are_rejected_before_any_launch():
  status, msg = call(search=1, k=1)                 # valid parameters, NULL device buffers
  assert status == -1 and "NULL" in msg, msg
  status, msg = call(scratch=16)
  assert status == -1 and "NULL" in msg, msg


def test_map_labels_argument_checks():
  lib = _lib.load()
  assert lib.pcls_map_labels(None, -1, None, 0, None, None) == -1
  assert b"pcls_map_labels" in lib.pcls_last_error()
  assert lib.pcls_map_labels(None, 10, None, 0, None, None) == -1
  assert b"NULL" in lib.pcls_last_error()
  assert lib.pcls_map_labels(None, 0, None, 0, None, None) == 0        # nothing to do
