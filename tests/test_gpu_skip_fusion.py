"""Skip fusion (option fuse_skip, Net::finalize): a 1x1 conv of the network input with no activation whose only reader adds
it after its ReLU (SqueezeSegV2's conv1_skip -> fire13's expand) is computed in that reader's epilogue from the 16-byte
input pixels (conv_tc.cu, RM = 3) instead of being written and read back as a 64-channel tensor.

The fused output is checked against a float64 evaluation with the fp16 error model of test_gpu_nets.py, against the same
graph built with fuse_skip = 0 (they may differ where the skip's fp32 sums round to different 16-bit values), and the
rule is checked not to fire where it must not."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import nn as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.nets import layers as L
from tests.test_gpu_nets import LOGIT_TOL, U16, TinyNet, _fold64, _input, _nchw, _rand_vars, _tp
from tests.util import synth_range_images

pytestmark = pytest.mark.gpu


def _graph(H, W, skip_act=False, second_reader=False):
  """conv1_skip (1x1 6 -> 64 + BN, no activation) and a fire13-like expand (16 -> 32 || 32, ReLU) that adds it."""
  t = TinyNet(H, W)
  g = t.g
  skip = L.BatchNormalization("bs")(L.Conv2D("cs", 64, 1)(g.input))
  if skip_act:
    skip = L.relu(skip)
  sq = L.relu(L.BatchNormalization("b1")(L.Conv2D("c1", 16, 3)(g.input)))
  e1 = L.relu(L.BatchNormalization("b2")(L.Conv2D("c2", 32, 1)(sq)))
  e3 = L.relu(L.BatchNormalization("b3")(L.Conv2D("c3", 32, 3)(sq)))
  out = L.add(L.concat([e1, e3]), skip)
  if second_reader:
    L.relu(L.Conv2D("cz", 16, 1)(skip))
  _rand_vars(g, np.random.default_rng(H * W))
  return t, sq, skip, out


def _run(t, out_sym, B, x, opts, keep=()):
  """-> (output, kept tensors, launches per forward, op names)"""
  lib = _lib.load()
  g = t.g
  opts = dict(opts, use_graph=0)
  if keep:
    opts["keep_tensors"] = 1
  net = g.build_net(t.logits, 2, 0, _lib.PCLS_F16, B, opts)
  stream = torch.cuda.current_stream().cuda_stream
  try:
    xd = torch.from_numpy(x).cuda()
    preds = torch.empty(x.shape[:3], dtype=torch.int32, device="cuda")
    _lib.check(lib.pcls_net_forward(net, xd.data_ptr(), 6, None, None, None, B, None, None, preds.data_ptr(), stream), "forward")
    res = []
    for sym in (out_sym,) + tuple(keep):
      o = torch.empty((B, g.H, sym.width, sym.channels), dtype=torch.float32, device="cuda")
      _lib.check(lib.pcls_net_read_tensor(net, sym.tid, B, o.data_ptr(), stream), "read_tensor")
      res.append(o)
    torch.cuda.synchronize()
    names = []
    for i in range(lib.pcls_net_num_ops(net)):
      buf, fam, fl, by = ctypes.create_string_buffer(64), ctypes.c_int(), ctypes.c_int64(), ctypes.c_int64()
      _lib.check(lib.pcls_net_op_info(net, i, buf, ctypes.byref(fam), ctypes.byref(fl), ctypes.byref(by)), "op_info")
      names.append((buf.value.decode(), by.value))
    return res[0].cpu().numpy(), [r.cpu().numpy() for r in res[1:]], lib.pcls_net_launches_per_forward(net), names
  finally:
    lib.pcls_net_destroy(net)


def _check_expand_plus_skip(x_dev, sq_dev, y_dev, p, what):
  """relu(expand(sq)) + skip(x) in float64 on the device's own 16-bit tensors.  Error model: the expand's and the
  skip's weights rounded to fp16 and their fp32 sums (1.5 x 2^-11 x S each), the activation and the skip each rounded to
  fp16 before the packed add (2^-11 x their magnitudes), the sum rounded once (2^-11 x |y|)."""
  ks, bs = _fold64(p, "cs", "bs")
  x = _nchw(x_dev).double()
  skip = O.conv2d_same(x, ks, bs)
  s_skip = O.conv2d_same(x.abs(), ks.abs(), bs.abs())
  q = _nchw(sq_dev).double()
  y_dev = _nchw(y_dev).double()
  worst = 0.0
  for conv, bn, sl in (("c2", "b2", slice(0, 32)), ("c3", "b3", slice(32, 64))):
    k, b = _fold64(p, conv, bn)
    act = torch.relu(O.conv2d_same(q, k, b))
    s = O.conv2d_same(q.abs(), k.abs(), b.abs())
    y = act + skip[:, sl]
    bound = U16 * (1.5 * (s + s_skip[:, sl]) + act + skip[:, sl].abs() + y.abs()) + 1e-6
    d = (y_dev[:, sl] - y).abs()
    worst = max(worst, float((d / bound).max()))
  assert worst <= 1.0, "%s: error %.3g x the fp16 error model" % (what, worst)
  return worst


@pytest.mark.parametrize("B", [1, 3, 32])
@pytest.mark.parametrize("W", [2048, 512, 256])
def test_fused_skip_against_oracle_and_unfused(W, B):
  """W = 2048 / 512: the expand runs the G = 4 pixel-group view, the rule fires.  W = 256: G = 2, it must not."""
  H = 2
  t, sq, skip, out = _graph(H, W)
  x = _input(np.random.default_rng(W + B), B, H, W)
  p = _tp(t.g)
  _, (ysq, yskip), _, _ = _run(t, out, B, x, {}, keep=(sq, skip))     # keep_tensors: un-fused, every tensor readable
  ref, _, n_ref, names_ref = _run(t, out, B, x, {"fuse_skip": 0})
  got, _, n_got, names_got = _run(t, out, B, x, {})
  fired = W >= 512
  assert not any(n.endswith("(fused)") and n.startswith("conv1x1_6x64") for n, _ in names_ref)
  assert any(n == "conv1x1_6x64_w%d(fused)" % W and by == 0 for n, by in names_got) == fired, names_got
  assert n_got == n_ref - (1 if fired else 0)
  _check_expand_plus_skip(x, ysq, ref, p, "fuse_skip = 0, W %d B %d" % (W, B))
  _check_expand_plus_skip(x, ysq, got, p, "fused, W %d B %d" % (W, B))
  if not fired:
    assert np.array_equal(got, ref)
    return
  # the two differ only where the skip's two fp32 sums (different order, bias split in two 16-bit parts) round to
  # different 16-bit values: at most one skip ulp plus the resulting rounding of the sum, on a tiny fraction of outputs
  d = np.abs(got - ref)
  n_diff = int((d > 0).sum())
  assert (d <= 2 * U16 * (np.abs(yskip) + np.abs(ref)) * 1.01 + 1e-7).all(), float(d.max())   # one ulp <= 2^-10 |v|
  assert n_diff <= 1e-3 * d.size, (n_diff, d.size)
  print("W %d B %d: %d of %d outputs differ from fuse_skip = 0 (max %.3g)" % (W, B, n_diff, d.size, float(d.max())))


@pytest.mark.parametrize("case", ["second_reader", "skip_activation", "keep_tensors", "conv_impl"])
def test_rule_does_not_fire(case):
  H, W, B = 2, 512, 2
  t, sq, skip, out = _graph(H, W, skip_act=case == "skip_activation", second_reader=case == "second_reader")
  x = _input(np.random.default_rng(5), B, H, W)
  opts = {"conv_impl": 1} if case == "conv_impl" else {}
  keep = (skip,) if case == "keep_tensors" else ()
  got, kept, n, names = _run(t, out, B, x, opts, keep=keep)
  ref, _, n_ref, _ = _run(t, out, B, x, dict(opts, fuse_skip=0), keep=keep)
  assert not any(name.endswith("(fused)") and name.startswith("conv1x1_6x64") for name, _ in names), names
  assert n == n_ref
  assert np.array_equal(got, ref)
  if keep:
    assert np.abs(kept[0]).max() > 0      # the skip tensor was written


def test_whole_squeezesegv2_fused_vs_unfused():
  """SqueezeSegV2 at the benchmark's shape (KITTI 64 x 2048, batch 32): conv1_skip is computed inside fire13's expand."""
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  H, W, B = 64, 2048, 32
  mc = config_map["squeezesegv2kitti"]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(11), B, H, W, valid_rate=0.78,
                                            num_classes=mc.NUM_CLASS)).cuda()
  out = {}
  for fuse in (1, 0):
    model = model_map["squeezesegv2"](mc)
    model.randomize_batch_norm(3)
    model.set_option("fuse_skip", fuse)
    res = model.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_logits=True)
    lib, net = _lib.load(), model._net
    names = []
    for i in range(lib.pcls_net_num_ops(net)):
      buf, fam, fl, by = ctypes.create_string_buffer(64), ctypes.c_int(), ctypes.c_int64(), ctypes.c_int64()
      _lib.check(lib.pcls_net_op_info(net, i, buf, ctypes.byref(fam), ctypes.byref(fl), ctypes.byref(by)), "op_info")
      names.append(buf.value.decode())
    out[fuse] = (res["logits"].cpu().numpy(), res["predictions"].cpu().numpy(), lib.pcls_net_launches_per_forward(net), names)
    del model
  (lg1, pd1, n1, names1), (lg0, pd0, n0, names0) = out[1], out[0]
  assert n1 == n0 - 1, (n1, n0)
  assert "conv1x1_6x64_w2048(fused)" in names1 and "conv1x1_6x64_w2048" in names0
  err = float(np.abs(lg1 - lg0).max())
  agree = float((pd1 == pd0).mean())
  print("SqueezeSegV2 64x2048 b32, fused vs fuse_skip = 0: logits max |d| %.3g, label agreement %.6f" % (err, agree))
  scale = max(1.0, float(np.abs(lg0).max()) / 4.0)
  assert err <= LOGIT_TOL * scale
  assert agree >= 0.9999
