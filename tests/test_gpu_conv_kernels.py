"""Every convolution kernel instantiation against float64, per op, at the tile counts the benchmark runs, in fp16 and bf16:

  conv_tc_kernel<T, KC, SUB, G, RES, LEAKY, KS, RM>   tcgen05 implicit GEMM (conv_tc.cu)
  pool_conv1x1_kernel<T, C, S>                       3x3 / [1,2] max-pool + 1x1 squeeze (pool_conv.cu)
  squeeze_upconv_kernel<T, C, S>                     1x1 squeeze + [1,4] / [1,2] transposed conv (squeeze_upconv.cu)

Each case is a small graph built with nets/layers.Graph (TinyNet of test_gpu_nets.py): c0 (3x3 conv of the network
input, BN, ReLU) makes the op's input, optional 1x1 convs make its residuals or its concat sibling, and the op under test
is the last op written.  Every case runs these checks:

  1. the op's output on every pixel of every frame against float64 (torch on the GPU) on the device's own 16-bit input,
     read back with keep_tensors = 1.  U = 2^-11 (fp16) / 2^-8 (bf16), S = sum |w'| |x| (+ |b'|), pre = conv + bias:
       fp32 epilogue (no residual; LeakyReLU or none with residuals; two residuals)  U (1.5 S + |y|)
       packed 16-bit add (ReLU + exactly one residual, epilogue_vec8)                U (1.5 S + relu(pre) + |y|)
       skip computed in the epilogue (RM = 3): the packed add, plus U (1.5 S_skip + |skip|) for the 16-bit skip
       pool_conv1x1: the exact 3x3 max of the input, then the fp32-epilogue model
       squeeze_upconv: the fp32-epilogue model on the un-fused squeeze tensor, slack 3.5 instead of 1.5 (the kernel's
       own squeeze values may differ from that tensor by one 16-bit ulp).
     Except for squeeze_upconv, each op is checked a second time against float64 with the weights as the device stores
     them (16-bit): the U S term of weight rounding drops out and K 2^-21 S (float32 accumulation of K terms, 8x its
     worst case) takes its place.  This bound sees a wrong rounding mode of the 16-bit conversions or packed adds;
  2. every element written: two forwards with different inputs, the second is checked (an element the second missed
     keeps the first one's value); a concat sibling written earlier in op order passes its own check;
  3. the same answer through other plumbing: a repeated forward and keep_tensors = 0 with CUDA-graph replays are
     bit-identical, and so is a micro-batched net (B = 7 with micro_batch = 3: the last pass has one frame);
  4. the kernel that ran (torch.profiler), with its template arguments, is the case's declared instantiation, and the
     launch count agrees with pcls_net_launches_per_forward;
  5. "wrap" cases reach >= 17 tiles per CTA (more than twice the largest accumulator count, 8): the second epilogue
     group, the accumulator parity flip, the bias pre-load of a later tile and the staging-buffer rotation all run.
     Counted conservatively from the shape: tiles >= ceil(Cout / 256) * frames * H * Wgemm / (128 G) over the SMs.

The census test profiles the benchmarked networks and requires every conv_tc_kernel instantiation they launch to be
declared by a wrap case here, and every pool_conv1x1 / squeeze_upconv instantiation by a benchmark-shape case.
"""
import ctypes
import re
import zlib

import numpy as np
import pytest
import torch

from oracle import nn as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.nets import layers as L
from tests.test_gpu_nets import TinyNet, _fold64, _input, _rand_vars, _tp

U = {"f16": 2.0 ** -11, "bf16": 2.0 ** -8}
PREC = {"f16": _lib.PCLS_F16, "bf16": _lib.PCLS_BF16}
FAMILY = {"tc": "conv_tc_kernel", "pc": "pool_conv1x1_kernel", "su": "squeeze_upconv_kernel"}
WRAP_TILES_PER_CTA = 17


def _case(cid, inst, op="conv", k=3, s=1, cin=64, cout=64, act="relu", res=0, src="a", H=64, W=1024, B=5, mb=0,
          regime="wrap", sib=False, merged=None, opts=None):
  """inst = (family, template arguments after T): ("tc", KC, SUB, G, RES, LEAKY, KS, RM), ("pc", C, S), ("su", C, S).
  op: conv | deconv | pool (max-pool + 1x1 S = cout) | up (1x1 to cout + transposed conv) | skip (RM = 3 graph);
  src: "a" (c0's output, cin channels) or "input" (the network input); sib: a 1x1 sibling writes the first cout channels
  of a concat before the op writes the rest; merged = (E1, E3): the op is a merged Fire expand 1x1 || 3x3."""
  return [pytest.param(dict(id=cid + "-" + prec, prec=prec, inst=inst, op=op, k=k, s=s, cin=cin, cout=cout, act=act,
                            res=res, src=src, H=H, W=W, B=B, mb=mb, regime=regime, sib=sib, merged=merged,
                            opts=opts or {}), id=cid + "-" + prec)
          for prec in ("f16", "bf16")]


def _small(**kw):
  return dict(H=8, W=256, B=2, regime=None, **kw)


CASES = [
    # ---- RM = 2: no residual, TMA-store epilogue ----
    *_case("rm2-g4-sub1", ("tc", 64, 1, 4, 0, 0, 4, 2), k=1, cin=16, W=2048, B=10),
    *_case("rm2-g4-sub3", ("tc", 64, 3, 4, 0, 0, 4, 2), cin=16, W=2048, B=10),
    *_case("rm2-g2-kc32", ("tc", 32, 3, 2, 0, 0, 2, 2), cin=16, cout=128, W=2048, B=5),
    *_case("rm2-g2-kc64", ("tc", 64, 1, 2, 0, 0, 4, 2), k=1, cin=32, cout=128, W=2048, B=5),
    *_case("rm2-g2-kc64-leaky", ("tc", 64, 1, 2, 0, 1, 4, 2), k=1, cin=32, act="leaky", W=2048, B=5),
    *_case("rm2-g1-kc16-sub1", ("tc", 16, 1, 1, 0, 0, 1, 2), k=1, cin=16, cout=192),
    *_case("rm2-g1-kc16-sub3-tail32", ("tc", 16, 3, 1, 0, 0, 1, 2), cin=16, cout=96),
    *_case("rm2-g1-kc32-sub1", ("tc", 32, 1, 1, 0, 0, 2, 2), k=1, cin=32, cout=192),
    *_case("rm2-g1-kc32-sub3-tail32", ("tc", 32, 3, 1, 0, 0, 2, 2), cin=32, cout=96),
    *_case("rm2-g1-kc64-sub1", ("tc", 64, 1, 1, 0, 0, 4, 2), k=1),
    *_case("rm2-g1-kc64-sub3", ("tc", 64, 3, 1, 0, 0, 4, 2)),
    *_case("rm2-kc16-5chunks", ("tc", 16, 1, 1, 0, 0, 1, 2), k=1, cin=80, **_small()),
    *_case("rm2-kc32-3chunks", ("tc", 32, 3, 1, 0, 0, 2, 2), cin=96, **_small()),
    *_case("rm0-kc64-2chunks-streamed", ("tc", 64, 3, 1, 0, 0, 4, 0), cin=128, **_small()),
    # fire6 / fire7's expand3x3 as planned: K-skip (48 channels in a 64-channel chunk), N-split across CTAs, 32-channel
    # tail block, writing the second half of a 384-channel concat after the expand1x1 sibling
    *_case("rm2-ks3-nsplit-tail-fire6-expand3x3", ("tc", 64, 3, 1, 0, 0, 3, 2), cin=48, cout=192, sib=True, W=128, B=40),
    # merged expand 64 -> 128 || 128: split-N per N tile, rows permuted so that each tile holds half of both parts
    *_case("rm2-nsplit-perm-merged-expand", ("tc", 64, 3, 1, 0, 0, 4, 2), merged=(128, 128), W=128, B=40),
    # ---- RM = 1: one TMA-loaded residual ----
    *_case("rm1-g4-relu", ("tc", 64, 3, 4, 1, 0, 4, 1), cin=16, res=1, W=2048, B=10),
    *_case("rm1-g4-leaky", ("tc", 64, 3, 4, 1, 1, 4, 1), cin=16, res=1, act="leaky", W=2048, B=10),
    *_case("rm1-g2-relu", ("tc", 64, 3, 2, 1, 0, 4, 1), cin=32, res=1, W=2048, B=5),
    *_case("rm1-g2-leaky", ("tc", 64, 3, 2, 1, 1, 4, 1), cin=32, res=1, act="leaky", W=2048, B=5),
    *_case("rm1-g1-relu", ("tc", 64, 3, 1, 1, 0, 4, 1), res=1),
    *_case("rm1-g1-leaky", ("tc", 64, 3, 1, 1, 1, 4, 1), res=1, act="leaky"),
    *_case("rm1-g1-relu-b7-micro_batch3", ("tc", 64, 3, 1, 1, 0, 4, 1), res=1, H=8, W=256, B=7, mb=3, regime=None),
    # ---- RM = 3: SqueezeSegV2's conv1_skip computed inside fire13's expand ----
    *_case("rm3-skip-fire13-expand", ("tc", 64, 3, 4, 1, 0, 4, 3), op="skip", cin=16, merged=(32, 32), W=2048, B=10),
    # ---- RM = 0: the generic kernel ----
    *_case("rm0-res-cpasync-direct-store", ("tc", 64, 3, 1, 1, 0, 4, 0), cout=32, res=1, W=512, B=10),
    *_case("rm0-res-per-chunk-loads-nnt2", ("tc", 64, 1, 1, 1, 1, 4, 0), k=1, cout=512, res=1, act="leaky", W=512),
    *_case("rm0-res-tma-1x1", ("tc", 64, 1, 1, 1, 0, 4, 0), k=1, cout=256, res=1),
    *_case("rm0-two-residuals", ("tc", 64, 3, 1, 1, 1, 4, 0), res=2, act="leaky"),
    *_case("rm0-direct-store-cout32", ("tc", 64, 3, 1, 0, 0, 4, 0), cout=32),
    *_case("rm0-direct-store-1x1-cout32", ("tc", 64, 1, 1, 0, 0, 4, 0), k=1, cout=32),
    *_case("rm0-direct-store-1x1-cout32-leaky", ("tc", 64, 1, 1, 0, 1, 4, 0), k=1, cout=32, act="leaky"),
    *_case("rm0-act-none-residual", ("tc", 64, 3, 1, 1, 0, 4, 0), res=1, act=None),
    # ---- Darknet's wide and strided shapes ----
    *_case("nnt2-1x1-512-streamed", ("tc", 64, 1, 1, 0, 1, 4, 2), k=1, cout=512, act="leaky", W=512),
    *_case("nnt4-1x1-1024-streamed", ("tc", 64, 1, 1, 0, 1, 4, 2), k=1, cout=1024, act="leaky", W=256),
    *_case("nnt2-3x3-512", ("tc", 64, 1, 1, 0, 1, 4, 2), cout=512, act="leaky", **_small()),
    *_case("deconv-two-phase-256", ("tc", 64, 1, 1, 0, 1, 4, 2), op="deconv", k=4, cout=256, act="leaky", W=512, B=10),
    *_case("s2-5d-view-cin64", ("tc", 64, 1, 1, 0, 1, 4, 2), s=2, act="leaky", W=2048),
    *_case("s2-pair-view-cin32", ("tc", 64, 3, 1, 0, 1, 4, 2), s=2, cin=32, act="leaky", W=2048),
    *_case("input-3x3-s2-pair", ("tc", 64, 3, 4, 0, 0, 4, 2), src="input", s=2, W=2048, B=20),
    *_case("input-3x3-s1-pair", ("tc", 64, 3, 4, 0, 1, 4, 2), src="input", cout=32, act="leaky", W=2048, B=20),
    *_case("input-1x1-pair", ("tc", 32, 1, 2, 0, 0, 2, 2), src="input", k=1, act=None, W=2048, B=10,
           opts={"fuse_skip": 0}),
    # ---- tile edges ----
    *_case("edge-w1000-not-multiple-of-bw", ("tc", 64, 3, 1, 0, 0, 4, 2), W=1000, B=6),
    *_case("edge-bw64-h63", ("tc", 64, 1, 1, 0, 0, 4, 2), H=63, W=48, B=110),
    *_case("edge-h1", ("tc", 64, 3, 1, 0, 0, 4, 2), H=1, W=2048, B=160),
    # ---- pool_conv1x1: all 10 (C, S); the benchmark's three at B = 32 ----
    *_case("pool-64-16-bench", ("pc", 64, 16), op="pool", cin=64, cout=16, H=64, W=1024, B=32, regime="bench"),
    *_case("pool-128-32-bench", ("pc", 128, 32), op="pool", cin=128, cout=32, H=64, W=512, B=32, regime="bench"),
    *_case("pool-256-48-bench", ("pc", 256, 48), op="pool", cin=256, cout=48, H=64, W=256, B=32, regime="bench"),
    *_case("pool-64-32", ("pc", 64, 32), op="pool", cin=64, cout=32, H=9, W=130, B=3, regime=None),
    *_case("pool-64-64", ("pc", 64, 64), op="pool", cin=64, cout=64, H=5, W=67, B=5, regime=None),
    *_case("pool-128-16", ("pc", 128, 16), op="pool", cin=128, cout=16, H=7, W=256, B=1, regime=None),
    *_case("pool-128-64", ("pc", 128, 64), op="pool", cin=128, cout=64, H=6, W=95, B=4, regime=None),
    *_case("pool-256-16", ("pc", 256, 16), op="pool", cin=256, cout=16, H=5, W=64, B=3, regime=None),
    *_case("pool-256-32", ("pc", 256, 32), op="pool", cin=256, cout=32, H=8, W=33, B=6, regime=None),
    *_case("pool-256-64", ("pc", 256, 64), op="pool", cin=256, cout=64, H=4, W=128, B=2, regime=None),
    # ---- squeeze_upconv: fire13 / fire12 / fire11 at the benchmark's widths, B = 32 ----
    *_case("up-64-16-fire13", ("su", 64, 16), op="up", cin=64, cout=16, H=64, W=1024, B=32, regime="bench"),
    *_case("up-128-16-fire12", ("su", 128, 16), op="up", cin=128, cout=16, H=64, W=512, B=32, regime="bench"),
    *_case("up-256-32-fire11", ("su", 256, 32), op="up", cin=256, cout=32, H=64, W=256, B=32, regime="bench"),
]


def _declared(regimes):
  return {(c.values[0]["inst"], c.values[0]["prec"]) for c in CASES if c.values[0]["regime"] in regimes}


def test_case_matrix_covers_every_pool_and_squeeze_upconv_instantiation():
  pc = {(i[1], i[2], p) for i, p in _declared(("bench", None)) if i[0] == "pc"}
  su = {(i[1], i[2], p) for i, p in _declared(("bench", None)) if i[0] == "su"}
  shapes = [(64, 16), (64, 32), (64, 64), (128, 16), (128, 32), (128, 64), (256, 16), (256, 32), (256, 48), (256, 64)]
  assert pc == {(c, s, p) for c, s in shapes for p in PREC} and len(pc) == 20
  assert su == {(c, s, p) for c, s in ((64, 16), (128, 16), (256, 32)) for p in PREC} and len(su) == 6
  bench = {(i[1], i[2]) for i, p in _declared(("bench",)) if i[0] == "pc"}
  assert bench == {(64, 16), (128, 32), (256, 48)}


# ---- graph ---------------------------------------------------------------------------------------------------------
def _conv(name, x, cout, k=1, s=1, act="relu", bn=True, kind="conv"):
  y = L.Conv2D(name, cout, k, strides=[1, s])(x) if kind == "conv" else L.Conv2DTranspose(name, cout)(x)
  if bn:
    y = L.BatchNormalization(name + "_bn")(y)
  return L.relu(y) if act == "relu" else L.LeakyReLU(0.1)(y) if act == "leaky" else y


class Case:
  """The graph of one case: `inp` is the op's input tensor as read back, `out` the tensor it writes, `res` the tensors
  it adds; checks = [(channel slice of `out`, reference function of the float64 inputs)]."""

  def __init__(self, c):
    self.c = c
    self.t = TinyNet(c["H"], c["W"])
    g = self.t.g
    g.merge_expand = c["merged"] is not None
    op, cin, cout = c["op"], c["cin"], c["cout"]
    self.res = []
    self.skip_src = None
    if op == "skip":
      self.skip_src = _conv("cs", g.input, 64, act=None)               # conv1_skip: 1x1 6 -> 64, BN, no activation
    src = g.input if c["src"] == "input" else _conv("c0", g.input, cin, 3)
    self.inp = src
    if op == "pool":
      self.out = _conv("op", L.max_pool2d(src), cout)
    elif op == "up":
      self.inp = _conv("sq", src, cout)
      self.out = _conv("op", self.inp, cout, kind="deconv", bn=False)
    else:
      for i in range(c["res"]):
        self.res.append(_conv("r%d" % i, src, cout))
      sib = _conv("sib", src, cout) if c["sib"] else None
      if c["merged"]:
        e1, e3 = c["merged"]
        y = L.concat([_conv("e1", src, e1, 1, act=c["act"]), _conv("e3", src, e3, 3, act=c["act"])])
      else:
        y = _conv("op", src, cout, c["k"], c["s"], c["act"], kind="deconv" if op == "deconv" else "conv")
      for r in self.res:
        y = L.add(y, r)
      if op == "skip":
        y = L.add(y, self.skip_src)
      self.out = L.concat([sib, y]) if sib is not None else y
    self.rng = np.random.default_rng(zlib.crc32(c["id"].encode()))
    _rand_vars(g, self.rng)
    self.p = {k: v.cuda() for k, v in _tp(g).items()}
    self.lib = _lib.load()

  @property
  def n_out(self):
    return sum(self.c["merged"]) if self.c["merged"] else self.c["cout"]

  def build(self, **opts):
    o = {"use_graph": 0, "keep_tensors": 0, "micro_batch": self.c["mb"]}
    o.update(self.c["opts"])
    o.update(opts)
    return _Net(self, o)


class _Net:
  def __init__(self, case, opts):
    self.case, self.lib = case, case.lib
    c = case.c
    self.h = case.t.g.build_net(case.t.logits, 2, 0, PREC[c["prec"]], c["B"], opts)
    mb = opts["micro_batch"]
    self.passes = -(-c["B"] // mb) if mb else 1
    self.last = c["B"] - (self.passes - 1) * mb if mb else c["B"]   # frames of the last pass (what read_tensor sees)

  def forward(self, x):
    B = self.case.c["B"]
    xd = torch.from_numpy(x).cuda()
    preds = torch.empty(x.shape[:3], dtype=torch.int32, device="cuda")
    _lib.check(self.lib.pcls_net_forward(self.h, xd.data_ptr(), 6, None, None, None, B, None, None, preds.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream), "pcls_net_forward")
    torch.cuda.synchronize()

  def read(self, sym):
    """The last pass's frames of `sym` as float32 NHWC on the GPU (the network input: its 6 real channels)."""
    g = self.case.t.g
    tid, ch = (0, 8) if sym.is_input else (sym.tid, sym.channels)
    o = torch.empty((self.last, g.H, sym.width, ch), dtype=torch.float32, device="cuda")
    _lib.check(self.lib.pcls_net_read_tensor(self.h, tid, self.last, o.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "pcls_net_read_tensor")
    torch.cuda.synchronize()
    return o[..., :6] if sym.is_input else o

  def close(self):
    self.lib.pcls_net_destroy(self.h)


# ---- check 1: float64 references -----------------------------------------------------------------------------------
def _nchw(t):
  return t.permute(0, 3, 1, 2).double()


def _fold_device(p, name, bn, transpose, prec):
  """The folded kernel and bias exactly as Net::add_conv stores them: BN folded in double (with the float32 epsilon the
  builder passes), the kernel rounded to float32 and then to the 16-bit type, the bias to float32."""
  k = p[name + "/kernel"].double()
  cout = k.shape[2] if transpose else k.shape[3]
  b = p[name + "/bias"].double() if (name + "/bias") in p else torch.zeros(cout, dtype=torch.float64, device=k.device)
  if bn:
    sc = p[bn + "/gamma"].double() / torch.sqrt(p[bn + "/moving_variance"].double() + float(np.float32(O.BN_EPS)))
    k = k * (sc.view(1, 1, -1, 1) if transpose else sc.view(1, 1, 1, -1))
    b = (b - p[bn + "/moving_mean"].double()) * sc + p[bn + "/beta"].double()
  t16 = torch.float16 if prec == "f16" else torch.bfloat16
  return k.float().to(t16).double(), b.float().double()


def _ref_conv(p, name, bn, x, k=3, s=1, transpose=False, prec=None):
  """(pre-activation, S, K) of one folded conv in float64 on the GPU; prec: with the device's 16-bit weights."""
  kk, b = _fold_device(p, name, bn, transpose, prec) if prec else _fold64(p, name, bn, transpose)
  kk, b = kk.cuda(), b.cuda()
  K = kk.numel() // b.numel() + 1                                        # products + bias per output
  if transpose:
    return O.conv2d_transpose_1x4_s2(x, kk, b), O.conv2d_transpose_1x4_s2(x.abs(), kk.abs(), b.abs()), K
  return O.conv2d_same(x, kk, b, (1, s)), O.conv2d_same(x.abs(), kk.abs(), b.abs(), (1, s)), K


def _act(pre, act):
  return torch.relu(pre) if act == "relu" else O.leaky(pre) if act == "leaky" else pre


def _assert_model(what, got, y, bound):
  d = (_nchw(got) - y).abs()
  r = d / bound
  worst = float(r.max())
  if worst > 1.0:
    i = np.unravel_index(int(r.argmax()), tuple(r.shape))
    raise AssertionError("%s: error %.3g x the error model, %d elements over; worst at (b, c, h, w) = %s: got %r, "
                         "float64 %r, bound %.3g" % (what, worst, int((r > 1).sum()), i, float(_nchw(got)[i]),
                                                     float(y[i]), float(bound[i])))
  return worst


def _check_values(case, out, inp, res, x_in):
  """Check 1 on every pixel of every frame read back.  out / inp / res / x_in: float32 NHWC GPU tensors.

  Each op is checked twice: with the float64 weights and the error model of the module docstring, and with the weights
  as the device stores them, where the weight rounding drops out and what remains is the float32 accumulation (allowed:
  K 2^-21 S, eight times the worst case of K sequential additions) and the 16-bit roundings of the epilogue (half an
  ulp each, <= U |v|).  The second bound sees a wrong rounding mode or a lost low-order term that the first one hides
  under U S."""
  c, p = case.c, case.p
  u = U[c["prec"]]
  x = _nchw(inp)
  act, cout = c["act"], c["cout"]
  if c["op"] == "up":
    pre, S, _ = _ref_conv(p, "op", None, x, transpose=True)
    y = torch.relu(pre)
    return _assert_model("squeeze + transposed conv", out, y, u * (3.5 * S + y.abs()) + 1e-6)

  def check(what, got, parts, act, adds=(), skip_bound=0.0):
    for prec in (None, c["prec"]):
      refs = [_ref_conv(p, *q, prec=prec) for q in parts]
      pre, S, K = torch.cat([r[0] for r in refs], 1), torch.cat([r[1] for r in refs], 1), max(r[2] for r in refs)
      y = _act(pre, act)
      bound = (1.5 * u if prec is None else K * 2.0 ** -21) * S + skip_bound
      if act == "relu" and len(adds) == 1:                               # packed 16-bit add: relu(pre) rounded first
        bound = bound + u * y
      for r in adds:
        y = y + r
      _assert_model("%s (%s weights)" % (what, "float64" if prec is None else "16-bit"), got, y,
                    bound + u * y.abs() + 1e-6)

  if c["op"] == "pool":
    pooled = O.max_pool_same(x, 3, (1, 2))                               # exact
    return check("max-pool + 1x1 %d -> %d" % (c["cin"], cout), out, [("op", "op_bn", pooled, 1)], act)
  off = 0
  if c["sib"]:                                                           # the sibling slice keeps its own values
    check("concat sibling (written first)", out[..., :cout], [("sib", "sib_bn", x, 1)], "relu")
    off = cout
  if c["merged"]:
    parts = [("e1", "e1_bn", x, 1), ("e3", "e3_bn", x, 3)]
  else:
    parts = [("op", "op_bn", x, c["k"], c["s"], c["op"] == "deconv")]
  adds = [_nchw(r) for r in res]
  skip_bound = 0.0
  if c["op"] == "skip":                                                  # the skip computed from the network input
    sk, s_sk, _ = _ref_conv(p, "cs", "cs_bn", _nchw(x_in), 1)
    adds.append(sk)
    skip_bound = u * (1.5 * s_sk + sk.abs())
  check("op", out[..., off:off + case.n_out], parts, act, adds, skip_bound)


# ---- check 4 / 5: kernel names and regime --------------------------------------------------------------------------
def _inst(name):
  """(family, is_bf16, template arguments after T) of a kernel name, demangled or mangled; None for other kernels."""
  for fam, k in FAMILY.items():
    n = 7 if fam == "tc" else 2
    m = re.search(k + r"<\s*([\w:]+)\s*," + r"\s*,".join([r"\s*([^,<>]+?)"] * n) + r"\s*>", name)
    if m:
      vals = [v.strip() for v in m.groups()[1:]]
      args = tuple(1 if v in ("true", "(bool)1") else 0 if v in ("false", "(bool)0") else int(v) for v in vals)
      return fam, "bfloat16" in m.group(1), args
    m = re.search(k + r"I(\w+?)" + "".join([r"L([ib])(\d+)E"] * n) + "E", name)
    if m:
      return fam, "bfloat16" in m.group(1), tuple(int(m.group(3 + 2 * i)) for i in range(n))
  assert not any(k in name for k in FAMILY.values()), "cannot read the template arguments of %r" % name
  return None


def _profiled(fn):
  """Runs fn under torch.profiler; returns the names of the CUDA kernels it launched, in launch order."""
  from torch.autograd import DeviceType
  from torch.profiler import ProfilerActivity, profile
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    fn()
    torch.cuda.synchronize()
  evs = [e for e in prof.events() if e.device_type == DeviceType.CUDA and "_kernel" in e.name]
  return [e.name for e in sorted(evs, key=lambda e: e.time_range.start)]


def _check_kernel(case, net, names):
  """Check 4: the op (the last conv-family launch of each pass) ran the declared instantiation; returns it."""
  c = case.c
  lpf = case.lib.pcls_net_launches_per_forward(net.h)
  assert len(names) == net.passes * lpf, "%d passes x %d launches expected, profiled %s" % (net.passes, lpf, names)
  got = None
  for i in range(net.passes):
    fams = [x for x in (_inst(n) for n in names[i * lpf:(i + 1) * lpf]) if x is not None]
    assert fams, names
    got = fams[-1]
    want = (c["inst"][0], c["prec"] == "bf16", tuple(c["inst"][1:]))
    assert got == want, "the op ran %s%s%s, the case declares %s" % (
        FAMILY[got[0]], "<bf16>" if got[1] else "<f16>", got[2], c["inst"])
  return got


def _check_regime(case, net, inst):
  c = case.c
  if c["regime"] != "wrap":
    return
  assert inst[0] == "tc"
  G = inst[2][2]
  frames = c["mb"] or c["B"]
  wgemm = c["W"] // 2 if (c["s"] == 2 or c["src"] == "input") else c["W"]   # pixel pairs; transposed: input columns
  tiles = -(-case.n_out // 256) * -(-frames * c["H"] * wgemm // (128 * G))
  sms = torch.cuda.get_device_properties(0).multi_processor_count
  assert tiles >= WRAP_TILES_PER_CTA * sms, "%d tiles on %d SMs: %.1f per CTA" % (tiles, sms, tiles / sms)


# ---- the per-op test -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES)
def test_conv_kernel_against_float64(c):
  case = Case(c)
  B, H, W = c["B"], c["H"], c["W"]
  x1, x2 = _input(case.rng, B, H, W), _input(case.rng, B, H, W)
  # keep_tensors switches the squeeze_upconv and skip fusions off: those run fused, their inputs come from a keep run
  fused = c["op"] in ("up", "skip")
  main = case.build(keep_tensors=0 if fused else 1)
  try:
    names = _profiled(lambda: main.forward(x1))
    inst = _check_kernel(case, main, names)
    _check_regime(case, main, inst)
    main.forward(x2)                                                     # check 2: the second forward is checked
    out = main.read(case.out)
    src = case.build(keep_tensors=1) if fused else main
    try:
      if fused:
        src.forward(x2)
      inp, res = src.read(case.inp), [src.read(r) for r in case.res]
      x_in = src.read(case.t.g.input) if case.skip_src is not None else None
    finally:
      if fused:
        src.close()
    _check_values(case, out, inp, res, x_in)
    del inp, res, x_in

    # ---- check 3: other plumbing ----
    main.forward(x2)
    assert torch.equal(main.read(case.out), out), "a repeated forward is not bit-identical"
    net = case.build(keep_tensors=0, use_graph=1)
    try:
      for i in range(3):                                                 # capture, then replays
        net.forward(x2)
        assert torch.equal(net.read(case.out), out), "keep_tensors = 0, use_graph = 1, call %d: outputs differ" % i
    finally:
      net.close()
    if B > 1:
      mb = 0 if c["mb"] else (B + 1) // 2
      net = case.build(keep_tensors=0 if fused else 1, micro_batch=mb)
      try:
        net.forward(x2)
        n = min(net.last, main.last)
        assert torch.equal(net.read(case.out)[-n:], out[-n:]), "micro_batch = %d: outputs differ" % mb
      finally:
        net.close()
  finally:
    main.close()


# ---- census of the benchmarked networks ----------------------------------------------------------------------------
def _bench_networks():
  import bench
  return sorted({(m, cfg, H, W) for m, cfg, H, W, _ in bench.WORKLOADS.values()})


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("net", _bench_networks(), ids=lambda n: "%s-%s-%dx%d" % n)
def test_census_every_shipped_instantiation_is_tested(net, prec):
  """Every kernel instantiation a benchmarked network launches (kernel choice does not depend on the batch: B = 1) is
  declared by a wrap-regime case (conv_tc_kernel) or a benchmark-shape case (pool_conv1x1 / squeeze_upconv) above."""
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  name, cfg, H, W = net
  mc = config_map[cfg]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  if name == "darknet21":
    mc.NUM_LAYERS = 21
  model = model_map[name](mc)
  model.precision = PREC[prec]
  model.set_option("use_graph", 0)
  x = torch.randn((1, H, W, 6), device="cuda")
  x[..., 5] = 1.0
  model.forward_device(x)                                                # build the net outside the profiled window
  names = _profiled(lambda: model.forward_device(x))
  used = {i for i in (_inst(n) for n in names) if i is not None}
  assert any(i[0] == "tc" for i in used), names
  want_bf16 = prec == "bf16"
  assert all(i[1] == want_bf16 for i in used), used
  declared = {(i[0], tuple(i[1:])) for i, p in _declared(("wrap",)) if p == prec and i[0] == "tc"}
  declared |= {(i[0], tuple(i[1:])) for i, p in _declared(("bench",)) if p == prec}
  missing = sorted((i[0], i[2]) for i in used if (i[0], i[2]) not in declared)
  assert not missing, "%s %s launches instantiations no wrap / benchmark-shape case declares: %s" % (name, prec, missing)
  model._release()


# ---- C ABI: a 16-bit output slice must be a whole number of 8-channel vectors --------------------------------------
@pytest.mark.gpu
def test_conv_cout_not_multiple_of_8_is_rejected():
  """cout = 20 into a 24-channel tensor: the tensor-core epilogue stores only whole 8-channel vectors (channels 16-19
  were left unwritten, the CUDA-core kernel wrote them), so pcls_net_conv rejects it; cout = 24 is accepted."""
  lib = _lib.load()
  h = ctypes.c_void_p()
  _lib.check(lib.pcls_net_create(ctypes.byref(h), 4, 64, _lib.PCLS_F16, 1), "pcls_net_create")
  keep = []

  def desc(cin, cout, k, src, dst):
    d = _lib.ConvDesc()
    w = np.full((k, k, cin, cout), 0.01, np.float32)
    keep.append(w)
    d.kind, d.kh, d.kw, d.stride_w, d.cin, d.cout = _lib.KIND_CONV, k, k, 1, cin, cout
    d.h_kernel = w.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    d.bn_eps, d.act, d.in_tensor, d.out_tensor = 1e-3, _lib.ACT_RELU, src, dst
    d.out_channel_offset, d.residual0, d.residual1, d.out_is_logits = 0, -1, -1, 0
    return d

  try:
    t1 = _lib.check(lib.pcls_net_tensor(h, 64, 32, 0), "pcls_net_tensor")
    t2 = _lib.check(lib.pcls_net_tensor(h, 64, 24, 0), "pcls_net_tensor")
    _lib.check(lib.pcls_net_conv(h, ctypes.byref(desc(6, 32, 3, 0, t1))), "conv 6 -> 32")
    assert lib.pcls_net_conv(h, ctypes.byref(desc(32, 20, 1, t1, t2))) == -1  # PCLS_ERR_INVALID
    assert b"multiple of 8" in lib.pcls_last_error()
    _lib.check(lib.pcls_net_conv(h, ctypes.byref(desc(32, 24, 1, t1, t2))), "conv 32 -> 24")
  finally:
    lib.pcls_net_destroy(h)
