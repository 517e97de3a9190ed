"""Network forward through the C ABI vs the fp32 CPU oracle: every op flavour in isolation (odd widths, asymmetric
SAME padding, concat offsets, residuals) and the three whole nets.

Tolerances (BASELINE.json north_star): logits max-abs error <= 1e-2 against the fp32 oracle for the 16-bit path,
argmax agreement >= 99.9 % of valid pixels."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import nn as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.nets import layers as L
from tests.util import synth_range_images

pytestmark = pytest.mark.gpu

LOGIT_TOL = 1e-2
IMPLS = [0, 1]  # conv_impl: 0 = tcgen05 implicit GEMM where the shape allows, 1 = CUDA-core direct kernel


def _f16(a):
  return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


class TinyNet:
  """One-op graphs built with the same Graph the model builders use."""

  def __init__(self, H, W):
    self.g = L.Graph(H, W)
    self.g.rng = np.random.default_rng(7)
    # the net needs a [B,H,W,NC] logits tensor: a throw-away 1x1 conv from the input, emitted FIRST so that the
    # tensor under test is the last thing written into the arena
    self.logits = L.Conv2D("zz_logits", 2, 1)(self.g.input)

  def run(self, out_sym, B, x6, conv_impl, keep=None):
    """Runs the graph; returns `out_sym` as float32 NHWC.  keep = list of further symbolic tensors to read back
    (self.kept, same order): the net is then built with keep_tensors = 1 (no arena reuse)."""
    lib = _lib.load()
    g = self.g
    opts = {"conv_impl": conv_impl, "use_graph": 0}
    if keep:
      opts["keep_tensors"] = 1
    for kv in os.environ.get("PCLS_TEST_OPTS", "").split(","):  # e.g. fuse_pool=0 (A/B experiments)
      if "=" in kv:
        opts[kv.split("=")[0]] = int(kv.split("=")[1])
    net = g.build_net(self.logits, 2, 0, _lib.PCLS_F16, B, opts)
    try:
      x = torch.from_numpy(x6).cuda()
      preds = torch.empty(x6.shape[:3], dtype=torch.int32, device="cuda")
      _lib.check(lib.pcls_net_forward(net, x.data_ptr(), 6, None, None, None, B, None, None, preds.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), "forward")
      out = torch.empty((B, g.H, out_sym.width, out_sym.channels), dtype=torch.float32, device="cuda")
      _lib.check(lib.pcls_net_read_tensor(net, out_sym.tid, B, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
      self.kept = []
      for sym in keep or []:
        if sym.is_input:    # the network input as the device stores it: 6 channels (+ 2 zero pad) in 16-bit
          k = torch.empty((B, g.H, g.W, 8), dtype=torch.float32, device="cuda")
          _lib.check(lib.pcls_net_read_tensor(net, 0, B, k.data_ptr(), torch.cuda.current_stream().cuda_stream))
          self.kept.append(k.cpu().numpy()[..., :6])
          continue
        k = torch.empty((B, g.H, sym.width, sym.channels), dtype=torch.float32, device="cuda")
        _lib.check(lib.pcls_net_read_tensor(net, sym.tid, B, k.data_ptr(), torch.cuda.current_stream().cuda_stream))
        self.kept.append(k.cpu().numpy())
      torch.cuda.synchronize()
      return out.cpu().numpy()
    finally:
      lib.pcls_net_destroy(net)


def _rand_vars(g, rng):
  for k, v in g.variables.items():
    if k.endswith("/kernel"):
      g.variables[k] = (rng.normal(size=v.shape) / np.sqrt(np.prod(v.shape[:-1]) / 2)).astype(np.float32)
    elif k.endswith("moving_variance"):
      g.variables[k] = rng.uniform(0.5, 1.5, v.shape).astype(np.float32)
    elif k.endswith("gamma"):
      g.variables[k] = rng.uniform(0.8, 1.2, v.shape).astype(np.float32)
    else:
      g.variables[k] = rng.normal(0, 0.2, v.shape).astype(np.float32)


def _input(rng, B, H, W):
  x = rng.normal(size=(B, H, W, 6)).astype(np.float32)
  x[..., 5] = rng.random((B, H, W)) < 0.8
  return _f16(x)


def _nchw(x):
  return torch.from_numpy(x).permute(0, 3, 1, 2).contiguous()


def _nhwc(t):
  return t.permute(0, 2, 3, 1).contiguous().numpy()


def _tp(g):
  return {k: torch.from_numpy(v) for k, v in g.variables.items()}


# ---- per-layer error model -------------------------------------------------------------------------------------
# Every conv op is checked at ITS OWN output against a float64 evaluation on the device's own 16-bit input tensor, so
# errors do not compound and the bound is the arithmetic's, not a fraction of the largest value:
#   folded weights are rounded to fp16            -> |d| <= 2^-11 * S,  S = sum |w'| |x| (+ |b'|)
#   fp32 accumulation of K = taps * Cin products  -> a fraction of 2^-11 * S for K <= ~10^3 (allowed: 0.5 * 2^-11 * S)
#   the stored output is rounded to fp16 once     -> |d| <= 2^-11 * |y|
# A wrong / misplaced tap weight changes the output by ~S / taps, two orders of magnitude above this bound.
U16 = 2.0 ** -11


def _fold64(p, conv, bn, transpose=False):
  """Folded float64 kernel (Keras layout) and bias of conv(+BN), like Net::add_conv."""
  k = p[conv + "/kernel"].double()
  cout = k.shape[2] if transpose else k.shape[3]
  b = p[conv + "/bias"].double() if (conv + "/bias") in p else torch.zeros(cout, dtype=torch.float64)
  if bn:
    sc = p[bn + "/gamma"].double() / torch.sqrt(p[bn + "/moving_variance"].double() + O.BN_EPS)
    k = k * (sc.view(1, 1, -1, 1) if transpose else sc.view(1, 1, 1, -1))
    b = (b - p[bn + "/moving_mean"].double()) * sc + p[bn + "/beta"].double()
  return k, b


def _check_layer(x_dev, y_dev, p, conv, bn=None, strides=(1, 1), act=None, transpose=False, residuals=(), what="", slack=1.5):
  """x_dev / y_dev / residuals: NHWC float32 arrays read back from the device (exact 16-bit values)."""
  k, b = _fold64(p, conv, bn, transpose)
  x = _nchw(x_dev).double()
  if transpose:
    pre = O.conv2d_transpose_1x4_s2(x, k, b)
    S = O.conv2d_transpose_1x4_s2(x.abs(), k.abs(), b.abs())
  else:
    pre = O.conv2d_same(x, k, b, strides)
    S = O.conv2d_same(x.abs(), k.abs(), b.abs(), strides)
  y = pre if act is None else (torch.relu(pre) if act == "relu" else O.leaky(pre))
  for r in residuals:
    y = y + _nchw(r).double()
  bound = U16 * (slack * S + y.abs()) + 1e-6
  d = (_nchw(y_dev).double() - y).abs()
  worst = float((d / bound).max())
  assert tuple(y.shape) == tuple(_nchw(y_dev).shape), what
  assert worst <= 1.0, "%s: error %.3g x the fp16 error model (max abs err %.3e)" % (what, worst, float(d.max()))
  return worst


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("H,W,c1,c2", [(5, 48, 32, 48), (3, 27, 16, 64), (8, 256, 64, 128), (2, 130, 128, 32)])
def test_conv_flavours_in_isolation(impl, H, W, c1, c2):
  """3x3 s1 from the 6-channel input, 1x1, 3x3 s[1,2] (asymmetric SAME for even W / symmetric for odd), transposed
  [1,4] s2, concat-by-offset (merged Fire expand) - each checked at its own output against the error model."""
  rng = np.random.default_rng(H * W + c1)
  B = 2
  t = TinyNet(H, W)
  g = t.g
  a = L.relu(L.BatchNormalization("b0")(L.Conv2D("c0", c1, 3)(g.input)))                      # 3x3 s1, Cin = 6
  b = L.LeakyReLU(0.1)(L.BatchNormalization("b1")(L.Conv2D("c1", c2, 1, use_bias=False)(a)))  # 1x1
  c = L.relu(L.Conv2D("c2", c1, 3, strides=[1, 2])(b))                                        # 3x3 s2, bias only
  d = L.relu(L.Conv2DTranspose("c3", c1)(c))                                                  # deconv back to >= W
  e1 = L.relu(L.BatchNormalization("b4")(L.Conv2D("c4", c2, 1)(d)))
  e3 = L.relu(L.BatchNormalization("b5")(L.Conv2D("c5", c2, 3)(d)))
  cat = L.concat([e1, e3])
  _rand_vars(g, rng)
  x = _input(rng, B, H, W)
  p = _tp(g)
  got = t.run(cat, B, x, impl, keep=[g.input, a, b, c, d])
  xin, ya, yb, yc, yd = t.kept
  assert np.array_equal(xin, x)                                      # the input was representable in fp16
  _check_layer(xin, ya, p, "c0", "b0", act="relu", what="3x3 s1 from the input")
  _check_layer(ya, yb, p, "c1", "b1", act="leaky", what="1x1")
  _check_layer(yb, yc, p, "c2", None, strides=(1, 2), act="relu", what="3x3 s[1,2]")
  _check_layer(yc, yd, p, "c3", None, act="relu", transpose=True, what="transposed [1,4] s[1,2]")
  _check_layer(yd, got[..., :c2], p, "c4", "b4", act="relu", what="expand1x1 (concat offset 0)")
  _check_layer(yd, got[..., c2:], p, "c5", "b5", act="relu", what="expand3x3 (concat offset c2)")


def F_relu(x):
  return torch.relu(x)


@pytest.mark.parametrize("W,cs,ce", [(512, 16, 64), (1024, 16, 32), (512, 32, 64), (256, 32, 128), (512, 16, 16),
                                     (128, 48, 192), (256, 64, 128)])
def test_wide_narrow_channel_layers(W, cs, ce):
  """The shapes of the benchmark's Fire layers (Cin = 16 / 32 at W >= 256: pixel-group view G = 4 / 2, banded MMA issue;
  Cin = 48 / 64 at W = 128 / 256: fire6-10), halo tiles, resident weights, split-N, TMA-store epilogue with the 5-D group
  map, residual prefetch and the single-pass transposed conv - each op against the error model at its own output."""
  rng = np.random.default_rng(W + cs + ce)
  B, H = 2, 3
  t = TinyNet(H, W)
  g = t.g
  a = L.relu(L.BatchNormalization("b0")(L.Conv2D("c0", 64, 3)(g.input)))                 # [W, 64] (pair view)
  skip = L.relu(L.BatchNormalization("bs")(L.Conv2D("cs", 2 * ce, 1)(a)))                # the tensor added at the end
  sq = L.relu(L.BatchNormalization("b1")(L.Conv2D("c1", cs, 1)(a)))                      # squeeze -> cs channels
  e1 = L.relu(L.BatchNormalization("b2")(L.Conv2D("c2", ce, 1)(sq)))                     # grouped 1x1
  e3 = L.relu(L.BatchNormalization("b3")(L.Conv2D("c3", ce, 3)(sq)))                     # grouped 3x3 (halo)
  cat = L.add(L.concat([e1, e3]), skip)                                                  # concat offsets + residual
  sq2 = L.relu(L.BatchNormalization("b4")(L.Conv2D("c4", cs, 1)(cat)))
  up = L.relu(L.Conv2DTranspose("c5", cs)(sq2))                                          # grouped single-pass deconv
  _rand_vars(g, rng)
  x = _input(rng, B, H, W)
  p = _tp(g)
  for impl in IMPLS:
    got = TinyNet.run(t, up, B, x, impl, keep=[g.input, a, skip, sq, cat, sq2])
    xin, ya, ys, yq, ycat, yq2 = t.kept
    _check_layer(xin, ya, p, "c0", "b0", act="relu", what="impl %d: 3x3 from the input" % impl)
    _check_layer(ya, ys, p, "cs", "bs", act="relu", what="impl %d: 1x1 64 -> 2ce" % impl)
    _check_layer(ya, yq, p, "c1", "b1", act="relu", what="impl %d: squeeze" % impl)
    _check_layer(yq, ycat[..., :ce], p, "c2", "b2", act="relu", residuals=[ys[..., :ce]], what="impl %d: expand1x1 + skip" % impl)
    _check_layer(yq, ycat[..., ce:], p, "c3", "b3", act="relu", residuals=[ys[..., ce:]], what="impl %d: expand3x3 + skip" % impl)
    _check_layer(ycat, yq2, p, "c4", "b4", act="relu", what="impl %d: squeeze 2" % impl)
    _check_layer(yq2, got, p, "c5", None, act="relu", transpose=True, what="impl %d: transposed conv" % impl)


@pytest.mark.parametrize("impl", IMPLS)
def test_residual_and_skip_adds(impl):
  rng = np.random.default_rng(3)
  B, H, W = 2, 4, 64
  t = TinyNet(H, W)
  g = t.g
  a = L.LeakyReLU(0.1)(L.BatchNormalization("b0")(L.Conv2D("c0", 32, 3, use_bias=False)(g.input)))
  s = L.LeakyReLU(0.1)(L.BatchNormalization("b1")(L.Conv2D("c1", 32, 1)(a)))
  y = L.LeakyReLU(0.1)(L.BatchNormalization("b2")(L.Conv2D("c2", 32, 3, use_bias=False)(s)))
  y += s          # block residual
  y = y + a       # encoder skip
  _rand_vars(g, rng)
  x = _input(rng, B, H, W)
  p = _tp(g)
  got = t.run(y, B, x, impl, keep=[g.input, a, s])
  xin, ya, ys = t.kept
  _check_layer(xin, ya, p, "c0", "b0", act="leaky", what="conv1")
  _check_layer(ya, ys, p, "c1", "b1", act="leaky", what="block 1x1")
  _check_layer(ys, got, p, "c2", "b2", act="leaky", residuals=[ys, ya], what="block 3x3 + residual + skip")


@pytest.mark.parametrize("C,S,W,H", [(64, 16, 256, 3), (64, 16, 70, 5), (128, 16, 33, 4), (256, 32, 14, 3), (128, 16, 15, 2)])
def test_squeeze_fused_into_transposed_conv(C, S, W, H):
  """squeeze_upconv_kernel: FIREUP's squeeze 1x1 conv (+BN, ReLU) and the [1,4] / stride [1,2] transposed conv (+bias,
  ReLU) behind it as one kernel (the squeeze tensor stays on chip).  Shapes of fire13 / fire12 / fire11, widths that are
  and are not multiples of the 14-pixel tile.  The un-fused run (keep_tensors switches the fusion off) gives the squeeze
  tensor; the fused output is checked against the error model on it.  The kernel's internal squeeze values may differ
  from that tensor by one 16-bit ulp where the accumulation order decides a rounding: 2 x 2^-11 x S more slack."""
  rng = np.random.default_rng(C + S + W)
  B = 2
  t = TinyNet(H, W)
  g = t.g
  a = L.relu(L.BatchNormalization("b0")(L.Conv2D("c0", C, 3)(g.input)))
  sq = L.relu(L.BatchNormalization("b1")(L.Conv2D("c1", S, 1)(a)))
  up = L.relu(L.Conv2DTranspose("c2", S, kernel_size=[1, 4], strides=[1, 2])(sq))
  _rand_vars(g, rng)
  x = _input(rng, B, H, W)
  p = _tp(g)
  ref = t.run(up, B, x, 0, keep=[a, sq])          # un-fused: two tcgen05 launches
  ya, ysq = t.kept
  _check_layer(ya, ysq, p, "c1", "b1", act="relu", what="squeeze %d -> %d" % (C, S))
  _check_layer(ysq, ref, p, "c2", None, act="relu", transpose=True, what="transposed conv (un-fused)")
  got = t.run(up, B, x, 0)                        # fused
  assert got.shape == ref.shape
  _check_layer(ysq, got, p, "c2", None, act="relu", transpose=True, slack=3.5, what="squeeze %d -> %d + transposed conv, fused" % (C, S))
  os.environ["PCLS_TEST_OPTS"] = "fuse_up=0"
  try:
    got2 = t.run(up, B, x, 0)
  finally:
    del os.environ["PCLS_TEST_OPTS"]
  assert np.array_equal(got2, ref)                # the switch restores the two-op path


@pytest.mark.parametrize("C,S,W,H", [(64, 16, 256, 9), (128, 32, 96, 20), (256, 48, 70, 5), (64, 16, 33, 3)])
def test_maxpool_fused_into_squeeze_conv(C, S, W, H):
  """pool_conv1x1_kernel: tf.nn.max_pool2d(3, [1,2], SAME) + the squeeze 1x1 conv behind it as one kernel (the pooled
  tensor never reaches memory).  Shapes of pool1 / pool3 / pool5 -> fire2 / fire4 / fire6 squeeze, even and odd widths,
  row segments; checked against the error model on the exact max-pool of the device's own input tensor, and against the
  un-fused path (fuse_pool = 0), which must give bit-identical results."""
  rng = np.random.default_rng(C + S + W)
  B = 2
  t = TinyNet(H, W)
  g = t.g
  a = L.relu(L.BatchNormalization("b0")(L.Conv2D("c0", C, 3)(g.input)))
  pooled = L.max_pool2d(a)
  sq = L.relu(L.BatchNormalization("b1")(L.Conv2D("c1", S, 1)(pooled)))
  out = L.relu(L.BatchNormalization("b2")(L.Conv2D("c2", 32, 1)(sq)))    # a consumer (reads the 48 -> 64 padded tensor too)
  _rand_vars(g, rng)
  x = _input(rng, B, H, W)
  p = _tp(g)
  got = t.run(out, B, x, 0, keep=[a, sq])
  ya, ysq = t.kept
  ypool = _nhwc(O.max_pool_same(_nchw(ya), 3, (1, 2)))
  _check_layer(ypool, ysq, p, "c1", "b1", act="relu", what="max-pool + squeeze %d -> %d" % (C, S))
  _check_layer(ysq, got, p, "c2", "b2", act="relu", what="consumer of the squeeze output")
  os.environ["PCLS_TEST_OPTS"] = "fuse_pool=0"
  try:
    got2 = t.run(out, B, x, 0, keep=[sq])
  finally:
    del os.environ["PCLS_TEST_OPTS"]
  _check_layer(ypool, t.kept[0], p, "c1", "b1", act="relu", what="un-fused reference path")
  assert np.abs(got2 - got).max() < 2e-2


def _report(name, cfg, H, W, B, impl, err, lmax, agree, agree_decidable):
  """Appends the measured parity numbers to gpurun_out/parity_report.jsonl (quoted in DESIGN.md)."""
  import json
  os.makedirs("gpurun_out", exist_ok=True)
  with open("gpurun_out/parity_report.jsonl", "a") as f:
    f.write(json.dumps(dict(model=name, config=cfg, H=H, W=W, B=B, conv_impl=impl, logits_max_abs_err=float(err),
                            logits_abs_max=lmax, label_agreement=agree,
                            label_agreement_decidable=agree_decidable)) + "\n")


def _model(name, cfg, H=None, W=None, seed=1):
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map[cfg]()
  if H:
    mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  model = model_map[name](mc)
  model.randomize_batch_norm(seed)
  return mc, model


def _oracle(mc, model, name, lidar, mask):
  arch = "squeezesegv2" if name == "squeezesegv2" else "darknet"
  return O.forward(arch, model.variables, lidar, mask, mc.CLASSES.index("None"),
                   num_layers=getattr(mc, "NUM_LAYERS", 53), output_stride=getattr(mc, "OUTPUT_STRIDE", 16))


def _prep(mc, raw):
  lidar, mask = [], []
  for b in range(raw.shape[0]):
    l, m, _ = O.input_stage(raw[b], mc.INPUT_MEAN, mc.INPUT_STD, mc.CLASSES.index("None"))
    lidar.append(l)
    mask.append(m)
  return np.stack(lidar), np.stack(mask)


@pytest.mark.parametrize("impl", IMPLS)
@pytest.mark.parametrize("name,cfg,H,W,B", [("squeezesegv2", "squeezesegv2", 32, 240, 3),
                                            ("squeezesegv2", "squeezesegv2kitti", 64, 512, 2),
                                            ("squeezesegv2", "squeezesegv2nuscenes", 32, 1024, 2),
                                            ("darknet21", "darknet21", 32, 240, 2),
                                            ("darknet53", "darknet53kitti", 64, 256, 1)])
def test_whole_net_logits_and_labels(impl, name, cfg, H, W, B):
  mc, model = _model(name, cfg, H, W)
  model.set_option("conv_impl", impl)
  rng = np.random.default_rng(1234)
  raw = synth_range_images(rng, B, H, W, valid_rate=0.78, num_classes=mc.NUM_CLASS)
  lidar, mask = _prep(mc, raw)
  lg_ref, pr_ref, pd_ref = _oracle(mc, model, name, lidar, mask)
  # (a) reference call contract: normalised [B,H,W,6] + bool mask, host arrays in, .numpy() out
  probs, preds = model([lidar, mask])
  assert tuple(probs.shape) == (B, H, W, mc.NUM_CLASS) and preds.dtype == torch.int32
  res = model.forward_device(torch.from_numpy(lidar).cuda(), torch.from_numpy(mask).cuda(), want_logits=True)
  lg = res["logits"].cpu().numpy()
  scale = max(1.0, float(np.abs(lg_ref).max()) / 4.0)   # tolerance is stated for O(1) logits
  err = np.abs(lg - lg_ref).max()
  assert err <= LOGIT_TOL * scale, "max abs logit error %g (scale %g)" % (err, scale)
  assert np.abs(probs.numpy() - pr_ref).max() <= err + 1e-6      # softmax is 1-Lipschitz in the max norm
  # label agreement (north star: >= 99.9 % of valid pixels).  A pixel whose two best oracle logits are closer than
  # twice the logits tolerance cannot be required to agree (the tolerance itself permits the flip), so the 99.9 % bar
  # is asserted on the decidable pixels and the raw agreement over ALL valid pixels must still be >= 99.8 %.
  same = preds.numpy() == pd_ref
  top2 = np.sort(lg_ref, axis=-1)[..., -2:]
  decidable = mask & ((top2[..., 1] - top2[..., 0]) > 2 * LOGIT_TOL * scale)
  agree = same[mask].mean()
  assert decidable.sum() > 0.5 * mask.sum()
  assert same[decidable].mean() >= 0.999, same[decidable].mean()
  assert agree >= 0.998, agree
  _report(name, cfg, H, W, B, impl, err, float(np.abs(lg_ref).max()), float(agree), float(same[decidable].mean()))
  assert (preds.numpy()[~mask] == mc.CLASSES.index("None")).all()
  # (b) raw input with the input stage fused into the first load gives the same predictions
  res2 = model.forward_device(torch.from_numpy(raw).cuda(), None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD,
                              want_logits=True)
  assert np.abs(res2["logits"].cpu().numpy() - lg).max() < 1e-3
  assert (res2["predictions"].cpu().numpy() == preds.numpy()).mean() > 0.9995
  # (c) predict_step contract
  p2, y2 = model.predict_step(((lidar, mask), None, None))
  assert np.array_equal(y2.numpy(), preds.numpy())


@pytest.mark.parametrize("name,cfg,H,W,B", [("squeezesegv2", "squeezesegv2nuscenes", 32, 1024, 2),
                                            ("darknet21", "darknet21", 32, 240, 2)])
def test_whole_net_bf16_storage(name, cfg, H, W, B):
  """The bf16 instantiation of every kernel (PCLS_BF16: bf16 storage, fp32 accumulation).  bf16 keeps 8 mantissa bits
  against fp16's 11, so the logits tolerance is 8x the fp16 one; labels must agree wherever the oracle's two best
  logits are further apart than twice that tolerance."""
  from pclsegmentation_b200 import _lib
  mc, model = _model(name, cfg, H, W)
  model.precision = _lib.PCLS_BF16
  model._release()
  rng = np.random.default_rng(77)
  raw = synth_range_images(rng, B, H, W, valid_rate=0.78, num_classes=mc.NUM_CLASS)
  lidar, mask = _prep(mc, raw)
  lg_ref, pr_ref, pd_ref = _oracle(mc, model, name, lidar, mask)
  res = model.forward_device(torch.from_numpy(lidar).cuda(), torch.from_numpy(mask).cuda(), want_logits=True)
  lg = res["logits"].cpu().numpy()
  scale = max(1.0, float(np.abs(lg_ref).max()) / 4.0)
  tol = 8 * LOGIT_TOL * scale
  err = np.abs(lg - lg_ref).max()
  assert err <= tol, "max abs logit error %g (tolerance %g)" % (err, tol)
  assert np.abs(res["probabilities"].cpu().numpy() - pr_ref).max() <= err + 1e-6
  same = res["predictions"].cpu().numpy() == pd_ref
  top2 = np.sort(lg_ref, axis=-1)[..., -2:]
  decidable = mask & ((top2[..., 1] - top2[..., 0]) > 2 * tol)
  assert decidable.sum() > 0.3 * mask.sum()
  assert same[decidable].mean() >= 0.999, same[decidable].mean()
  assert same[mask].mean() >= 0.98, same[mask].mean()
  _report(name + "/bf16", cfg, H, W, B, 0, err, float(np.abs(lg_ref).max()), float(same[mask].mean()),
          float(same[decidable].mean()))


def test_micro_batch_and_graph_replay_are_equivalent():
  mc, model = _model("squeezesegv2", "squeezesegv2", 32, 240)
  rng = np.random.default_rng(2)
  raw = synth_range_images(rng, 5, 32, 240, num_classes=11)
  lidar, mask = _prep(mc, raw)
  model.set_option("use_graph", 0)
  base = model.forward_device(torch.from_numpy(lidar).cuda(), torch.from_numpy(mask).cuda(), want_logits=True)
  base = {k: v.clone() for k, v in base.items()}
  for opts in ({"use_graph": 1}, {"micro_batch": 2, "use_graph": 1}, {"micro_batch": 2, "use_graph": 0}):
    for k, v in opts.items():
      model.set_option(k, v)
    for _ in range(3):  # replays
      out = model.forward_device(torch.from_numpy(lidar).cuda(), torch.from_numpy(mask).cuda(), want_logits=True)
    assert torch.equal(out["predictions"], base["predictions"]) and torch.equal(out["logits"], base["logits"])


@pytest.mark.parametrize("channels,with_mask", [(6, True), (6, False), (8, True), (8, False)])
def test_16bit_host_input_gives_identical_results(channels, with_mask):
  """model([lidar.astype(float16), mask]) - the 12 / 16 bytes-per-pixel host contract (pcls_net_forward_in16) - must be
  bit-identical to the float32 call: the device rounds the float32 input to the same 16-bit values first."""
  mc, model = _model("squeezesegv2", "squeezesegv2", 32, 240)
  rng = np.random.default_rng(11)
  raw = synth_range_images(rng, 5, 32, 240, num_classes=11)
  lidar, mask = _prep(mc, raw)
  base = model.forward_device(torch.from_numpy(lidar).cuda(), torch.from_numpy(mask).cuda(), want_logits=True)
  base = {k: v.clone() for k, v in base.items()}
  l16 = lidar.astype(np.float16)
  if channels == 8:
    l16 = np.concatenate([l16, rng.standard_normal(l16.shape[:3] + (2,)).astype(np.float16)], -1)  # pads are ignored
  m = torch.from_numpy(mask).cuda() if with_mask else None
  for _ in range(2):  # capture + replay
    out = model.forward_device(torch.from_numpy(l16).cuda(), m, want_logits=True)
  assert torch.equal(out["logits"], base["logits"]) and torch.equal(out["predictions"], base["predictions"])
  assert torch.equal(out["probabilities"], base["probabilities"])
  # through the reference-facing call with host arrays, micro-batched (the pointer must walk 2-byte elements)
  model.set_option("micro_batch", 2)
  probabilities, predictions = model([l16, mask if with_mask else None])
  assert np.array_equal(predictions.numpy(), base["predictions"].cpu().numpy())
  with pytest.raises(ValueError):
    model.forward_device(torch.from_numpy(l16).cuda().to(torch.bfloat16), m)
