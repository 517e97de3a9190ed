"""Test-time augmentation without a GPU: the oracle's view and merge rules (oracle/tta.py), the ``TTA`` spec and the
argument checks of pcls_tta_views / pcls_tta_merge."""
import ctypes
import itertools

import numpy as np
import pytest

from oracle import tta as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.tta import TTA, from_args, parse_shifts, view_rotation
from tests.util import synth_range_images


@pytest.mark.parametrize("W", [8, 12, 30, 2048])
def test_view_then_inverse_is_identity(W):
  for flip, shift in itertools.product((0, 1), sorted({0, 1, W // 4, W // 2, W - 1, 7 % W})):
    fwd, inv = O.columns(flip, shift, W), O.inverse_columns(flip, shift, W)
    assert sorted(fwd) == list(range(W))
    assert np.array_equal(inv[fwd], np.arange(W)) and np.array_equal(fwd[inv], np.arange(W))


@pytest.mark.parametrize("W", [8, 30, 2048])
def test_mirror_twice_and_rolls_compose(W):
  mirror = O.columns(1, 0, W)
  assert np.array_equal(mirror[mirror], np.arange(W))
  for a, b in itertools.product((0, 1, 5 % W, W // 2, W - 1), repeat=2):
    ra, rb = O.columns(0, a, W), O.columns(0, b, W)
    assert np.array_equal(rb[ra], O.columns(0, (a + b) % W, W))
  # the mirror first, then the roll
  for s in (1, W // 2, W - 1):
    assert np.array_equal(O.columns(0, s, W)[mirror], O.columns(1, s, W))


def test_quarter_turns_are_exact():
  W = 2048
  for k, (c, s) in enumerate(((1.0, 0.0), (0.0, -1.0), (-1.0, 0.0), (0.0, 1.0))):
    assert O.rotation(k * W // 4, W) == (c, s) == view_rotation(k * W // 4, W)
  x = np.array([1.5, -2.25, 3e7, -0.0], np.float32)
  y = np.array([0.5, 7.0, -1e-3, 4.0], np.float32)
  xd, yd = O.view_points(x, y, 0, W // 2, W)
  assert np.array_equal(xd, -x.astype(np.float64)) and np.array_equal(yd, -y.astype(np.float64))
  xd, yd = O.view_points(x, y, 0, W // 4, W)          # alpha = -pi/2: (x, y) -> (y, -x)
  assert np.array_equal(xd, y.astype(np.float64)) and np.array_equal(yd, -x.astype(np.float64))
  xd, yd = O.view_points(x, y, 1, 0, W)
  assert np.array_equal(np.signbit(yd), ~np.signbit(y)) and np.array_equal(xd, x.astype(np.float64))
  # a general shift: the rotation is the float64 one, not a quarter turn
  c, s = view_rotation(5, W)
  assert c == pytest.approx(np.cos(-2 * np.pi * 5 / W), abs=0) and s < 0


def test_rotation_matches_the_projection_columns():
  """A point's view column is where the projection would put the rotated / mirrored point (away from boundaries)."""
  W = 2048
  rng = np.random.default_rng(0)
  yaw = rng.uniform(-np.pi, np.pi, 2000)
  x, y = np.cos(yaw) * 10, np.sin(yaw) * 10

  def col(x, y):
    p = 0.5 * (-np.arctan2(y, x) / np.pi + 1.0) * W
    return np.floor(p).astype(np.int64) % W, p

  c0, p0 = col(x, y)
  keep = np.abs(p0 - np.round(p0)) > 1e-3
  for flip, shift in ((1, 0), (0, 1), (0, 512), (0, 1024), (1, 1537), (0, 333)):
    xd, yd = O.view_points(x.astype(np.float32), y.astype(np.float32), flip, shift, W)
    c1, _ = col(xd, yd)
    assert np.array_equal(c1[keep], O.columns(flip, shift, W)[c0[keep]]), (flip, shift)


def test_view_zero_is_the_plain_input_stage():
  from oracle import nn as onn
  rng = np.random.default_rng(1)
  raw = synth_range_images(rng, 2, 4, 16)
  raw[0, 0, 0, :2] = [-0.0, -0.0]
  mean, std = np.array([10.0, 0.0, -1.0, 0.2, 12.0]), np.array([12.0, 9.0, 1.5, 0.15, 12.5])
  got, mask = O.views_input(raw, mean, std, [(0, 0)], "f16")
  for b in range(2):
    lid, msk, _ = onn.input_stage(raw[b], mean, std, 0)
    f = np.zeros(lid.shape[:-1] + (8,), np.float32)
    f[..., :6] = lid
    assert np.array_equal(got[b], f.astype(np.float16).view(np.uint16))
    assert np.array_equal(mask[b], msk.astype(np.uint8))


def test_views_input_permutes_the_mask():
  rng = np.random.default_rng(2)
  raw = synth_range_images(rng, 3, 5, 24, channels=5)
  views = [(0, 0), (1, 0), (0, 7), (1, 12)]
  inp, mask = O.views_input(raw, np.zeros(5), np.ones(5), views, "bf16")
  for t, (f, s) in enumerate(views):
    inv = O.inverse_columns(f, s, 24)
    assert np.array_equal(mask[t * 3:(t + 1) * 3], (raw[..., 4] > 0)[:, :, inv])
    # channel 2 (z) moves with the column but keeps its value; empty pixels are zeros (not -0)
    z = np.where(raw[..., 4] > 0, raw[..., 2], np.float32(0))
    assert np.array_equal(inp[t * 3:(t + 1) * 3, ..., 2], O.to16(z, "bf16")[:, :, inv])


def test_merge_rules():
  rng = np.random.default_rng(3)
  T, B, H, W, NC = 3, 2, 2, 8, 5
  views = [(0, 0), (1, 3), (0, 5)]
  probs = rng.random((T * B, H, W, NC)).astype(np.float32)
  mask = np.ones((T * B, H, W), np.uint8)
  mask[0, 0, 2] = 0                                    # view 0 is the identity: source pixel (0, 0, 2) is empty
  mean, pred = O.merge(probs, mask, views, none_index=4)
  want = np.zeros((B, H, W, NC), np.float32)
  for t, (f, s) in enumerate(views):
    p = probs[t * B:(t + 1) * B][:, :, O.columns(f, s, W)]
    want = p if t == 0 else (want + p).astype(np.float32)
  assert np.array_equal(mean, want / np.float32(T))
  assert pred[0, 0, 2] == 4 and (pred != 4).sum() > 0
  # T = 1 returns p_0 unchanged, also under a non-identity view
  p1, _ = O.merge(probs[:B], mask[:B], [(1, 2)], 0)
  assert np.array_equal(p1, probs[:B][:, :, O.columns(1, 2, W)])
  # ties go to the first index; a NaN never wins
  tie = np.array([[[[0.25, 0.5, 0.5, 0.25]]]], np.float32)
  assert O.argmax_first(tie)[0, 0, 0] == 1
  assert O.argmax_first(np.array([np.nan, 0.1, 0.1], np.float32))[()] == 1


def test_tta_spec():
  assert TTA().view_list == [(0, 0), (1, 0)]
  assert TTA(flip=True, shifts=(0, 1024)).view_list == [(0, 0), (0, 1024), (1, 0), (1, 1024)]
  assert TTA(flip=False, shifts=(5, 0)).view_list == [(0, 5), (0, 0)]
  f, s, c, sn = TTA(shifts=(0, 512)).views(2048)
  assert f.tolist() == [0, 0, 1, 1] and s.tolist() == [0, 512, 0, 512]
  assert c.tolist() == [1.0, 0.0, 1.0, 0.0] and sn.tolist() == [0.0, -1.0, 0.0, -1.0]
  assert len(TTA(shifts=(0, 1, 2, 3))) == 8
  with pytest.raises(ValueError, match="at most 8"):
    TTA(shifts=(0, 1, 2, 3, 4))
  with pytest.raises(ValueError, match="twice"):
    TTA(shifts=(3, 3))
  with pytest.raises(ValueError, match=">= 0"):
    TTA(shifts=(-1,))
  with pytest.raises(ValueError, match="not in"):
    TTA(shifts=(0, 2048)).views(2048)
  assert parse_shifts("0,1024") == (0, 1024)
  assert from_args(False, None) is None
  assert from_args(True, None).view_list == [(0, 0), (1, 0)]
  assert from_args(False, "0,7").view_list == [(0, 0), (0, 7)]


def _views_call(lib, n=2, flip=(0, 1), shift=(0, 3), channels=5, W=8, cos_=(1.0, 0.5), mean=True, raw=1, out=1):
  arr = lambda t, v: (t * len(v))(*v)
  m5 = arr(ctypes.c_double, [0.0] * 5) if mean else None
  return lib.pcls_tta_views(raw, channels, 1, 4, W, m5, arr(ctypes.c_double, [1.0] * 5), n, arr(ctypes.c_int, flip),
                            arr(ctypes.c_int, shift), arr(ctypes.c_double, cos_), arr(ctypes.c_double, [0.0] * len(cos_)),
                            0, out, out, None)


def _merge_call(lib, n=2, flip=(0, 1), shift=(0, 3), nc=20, none=0, W=8, preds=1):
  arr = lambda t, v: (t * len(v))(*v)
  return lib.pcls_tta_merge(1, 1, 1, 4, W, nc, none, n, arr(ctypes.c_int, flip), arr(ctypes.c_int, shift), None, preds,
                            None)


def test_argument_validation_without_gpu():
  lib = _lib.load()
  for kw, msg in ((dict(n=0, flip=(), shift=(), cos_=()), b"n_views"),
                  (dict(n=9, flip=(0,) * 9, shift=tuple(range(9)), cos_=(1.0,) * 9, W=16), b"n_views"),
                  (dict(flip=(0, 0), shift=(3, 3)), b"same"),
                  (dict(shift=(0, 8)), b"shift 8"),
                  (dict(shift=(-1, 0)), b"shift -1"),
                  (dict(flip=(0, 2)), b"flip 2"),
                  (dict(channels=4), b"channels"),
                  (dict(channels=8), b"channels"),
                  (dict(mean=False), b"NULL"),
                  (dict(raw=None), b"NULL"),
                  (dict(out=None), b"NULL"),
                  (dict(cos_=(1.0, float("nan"))), b"finite")):
    assert _views_call(lib, **kw) == -1, kw
    assert b"pcls_tta_views" in lib.pcls_last_error() and msg in lib.pcls_last_error(), (kw, lib.pcls_last_error())
  for kw, msg in ((dict(n=0, flip=(), shift=()), b"n_views"),
                  (dict(n=9, flip=(0,) * 9, shift=tuple(range(9)), W=16), b"n_views"),
                  (dict(flip=(1, 1), shift=(3, 3)), b"same"),
                  (dict(shift=(0, 8)), b"shift 8"),
                  (dict(nc=33), b"num_classes"),
                  (dict(nc=0), b"num_classes"),
                  (dict(none=20), b"none_index"),
                  (dict(preds=None), b"NULL")):
    assert _merge_call(lib, **kw) == -1, kw
    assert b"pcls_tta_merge" in lib.pcls_last_error() and msg in lib.pcls_last_error(), (kw, lib.pcls_last_error())
