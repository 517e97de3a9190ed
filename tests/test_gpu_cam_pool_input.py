"""The CAM, the stand-alone max-pool and the network-input kernels per op, in fp16 and bf16:

  cam2_kernel<T, C>            CAM (nets/SqueezeSegV2.py), C = 64 / 128, row segments on blockIdx.z (nn_kernels.cu)
  maxpool3x3_s2_kernel<T>      3x3 / [1,2] SAME max-pool, row segments on blockIdx.y
  net_input_kernel<T>          float32 input -> tensor 0 + mask (normalised, or raw with the input stage fused)
  net_input16_kernel           16-bit input -> tensor 0 + mask (pcls_net_forward_in16)

CAM cases are graphs built with nets/layers.Graph (TinyNet of test_gpu_nets.py): c0 (3x3 conv of the network input,
BN, then ReLU, or no activation for the signed cases) makes the CAM's input; in pool cases a max-pool of the CAM's output
is the graph's last op.  Every CAM case runs these checks:

  1. every pixel of every frame against float64 (torch on the GPU) on the device's own 16-bit input, read back with
     keep_tensors = 1, with the error model of _check_cam; the max-pool behind it must equal the exact max-pool of the
     CAM output it read;
  2. every element written: two forwards with different inputs, the second is checked;
  3. the same answer through other plumbing: a repeated forward and keep_tensors = 0 with CUDA-graph replays are
     bit-identical, and so is the same input through a different row-segment plan (micro_batch = 1 for B > 1, a batch
     of three copies for B = 1): each pixel's arithmetic does not depend on the plan;
  4. the kernel that ran is cam2_kernel<T, C> (torch.profiler), the launch count agrees with
     pcls_net_launches_per_forward, and the kernel's grid is the one _cam_plan (a copy of launch_cam's segment choice)
     gives for the device's SM count;
  5. the case matrix reaches, at 148 SMs, every segment count 1-8 for each C and precision, a last segment shorter than
     the others, a last segment shorter than the 7-row window, H < 7 and signed input (test_cam_case_matrix, no GPU).

The max-pool is checked for exact equality with O.max_pool_same on its own input, on signed inputs (only -inf padding
gives the right answer), odd and even widths, several row segments and a short last one; both as the graph's last op
and in front of a 1x1 conv with fuse_pool = 0.

The input kernels are checked bit for bit against numpy / torch chains of round-to-nearest-even conversions (tensor 0
read raw through pcls_net_input_buffers), above the kernels' grid cap of sm_count * 16 * 256 pixels, and on the
mask-channel edges, where both entry points must agree pixel by pixel.

The census test profiles every benchmarked network and requires each pcls:: kernel it launches to be owned by a
per-op test: this file, test_gpu_conv_kernels.py or test_gpu_logits_head.py.
"""
import csv
import ctypes
import json
import os
import re
import tempfile
import zlib

import numpy as np
import pytest
import torch

from oracle import nn as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.nets import layers as L
from tests import test_gpu_conv_kernels as CK
from tests import test_gpu_logits_head as LH
from tests.test_gpu_nets import TinyNet, _fold64, _input, _rand_vars, _tp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = {"f16": 2.0 ** -11, "bf16": 2.0 ** -8}
SUB = {"f16": 2.0 ** -25, "bf16": 2.0 ** -134}   # half the smallest subnormal: the absolute rounding error near zero
TANH = 2.0 ** -10                                # tanh.approx.f32: a margin over its relative error of 2^-11
PREC = {"f16": _lib.PCLS_F16, "bf16": _lib.PCLS_BF16}
DT = {"f16": torch.float16, "bf16": torch.bfloat16}
TNAME = {"f16": "__half", "bf16": "__nv_bfloat16"}
CAM_CTAS = 3                                     # nn_kernels.cu: resident CAM CTAs per SM the plan assumes
REF_SMS = 148                                    # B200


# ---- launch plans: copies of launch_cam / launch_maxpool3x3_s2 / launch_net_input ---------------------------------
def _cam_plan(C, B, H, W, sms):
  """(grid, rows per segment, rows of the last segment) of cam2_kernel, as launch_cam chooses them."""
  TW = 256 // (C // 8)
  strips, slots = -(-W // TW) * B, sms * CAM_CTAS
  segs, best = 1, None
  for s in range(1, (H // 8 if H >= 8 else 1) + 1):
    cost = -(-strips * s // slots) * (-(-H // s) + 7)
    if best is None or cost < best:
      best, segs = cost, s
  rps = -(-H // segs)
  segs = -(-H // rps)
  return (-(-W // TW), B, segs), rps, H - (segs - 1) * rps


def _pool_plan(C, B, H, Win, sms):
  Wout = (Win + 1) // 2
  n_cols = B * Wout * (C // 8)
  segs = max(min(-(-sms * 2048 * 2 // n_cols), H // 8), 1)
  rps = -(-H // segs)
  segs = -(-H // rps)
  return (-(-n_cols // 256), segs, 1), rps, H - (segs - 1) * rps


def _input_grid(n_pixels, sms):
  return (min(-(-n_pixels // 256), sms * 16), 1, 1)


def _sms():
  return torch.cuda.get_device_properties(0).multi_processor_count


# ---- profiling: kernel names and grids from the chrome trace -------------------------------------------------------
def _trace(fn):
  """Runs fn under torch.profiler; returns [(kernel name, grid)] in launch order, from the exported chrome trace."""
  from torch.profiler import ProfilerActivity, profile
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    fn()
    torch.cuda.synchronize()
  with tempfile.TemporaryDirectory() as d:
    path = os.path.join(d, "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
      evs = json.load(f)["traceEvents"]
  ks = sorted((e for e in evs if e.get("cat") == "kernel" and "_kernel" in e.get("name", "")), key=lambda e: e["ts"])
  out = []
  for e in ks:
    g = e.get("args", {}).get("grid")
    assert g is not None, "the profiler trace records no grid for %s" % e["name"]
    out.append((e["name"], tuple(int(v) for v in g)))
  return out


def _cam_inst(name):
  """(T, C) of a cam2_kernel name, demangled or mangled; None for other kernels."""
  m = re.search(r"cam2_kernel<\s*([\w:]+)\s*,\s*(\d+)\s*>", name) or re.search(r"cam2_kernelI(\d+\w+?)Li(\d+)EE", name)
  if not m:
    return None
  return ("__nv_bfloat16" if "bfloat16" in m.group(1) else "__half"), int(m.group(2))


def _tmpl(name, kernel):
  """T of a kernel<T> name, demangled or mangled; None if `name` is not that kernel."""
  m = re.search(kernel + r"<\s*([\w:]+)\s*>", name) or re.search(kernel + r"I(\w+?)EEv", name)
  if not m:
    return None
  return "__nv_bfloat16" if "bfloat16" in m.group(1) else "__half"


def _check_launches(lib, h, passes, trace):
  lpf = lib.pcls_net_launches_per_forward(h)
  assert len(trace) == passes * lpf, "%d passes x %d launches expected, profiled %s" % (passes, lpf, trace)


# ---- device views ---------------------------------------------------------------------------------------------------
class _DevArray:
  """A raw device pointer as a __cuda_array_interface__ (torch.as_tensor reads it without a copy)."""

  def __init__(self, ptr, shape, typestr):
    self.__cuda_array_interface__ = dict(shape=tuple(shape), typestr=typestr, data=(int(ptr), False), version=3)


def _input_buffers(lib, h, B, H, W):
  """(tensor 0 as raw int16 bits [B,H,W,8], mask buffer [B,H,W] u8), copies of the last pass."""
  inp, msk, frames = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int()
  _lib.check(lib.pcls_net_input_buffers(h, ctypes.byref(inp), ctypes.byref(msk), ctypes.byref(frames)),
             "pcls_net_input_buffers")
  assert B <= frames.value
  torch.cuda.synchronize()
  t0 = torch.as_tensor(_DevArray(inp.value, (B, H, W, 8), "<i2"), device="cuda").clone()
  m = torch.as_tensor(_DevArray(msk.value, (B, H, W), "|u1"), device="cuda").clone()
  return t0, m


def _bits(t, prec):
  """16-bit patterns of a float tensor rounded to the storage type (round to nearest even)."""
  return t.to(DT[prec]).view(torch.int16)


def _same16(a, b, prec):
  """Bit-identical, except that any NaN equals any NaN (the payload of a converted NaN is not specified)."""
  fa, fb = a.view(DT[prec]), b.view(DT[prec])
  return (a == b) | (torch.isnan(fa) & torch.isnan(fb))


# ---- CAM error model ------------------------------------------------------------------------------------------------
def _check_cam(x_dev, y_dev, p, name, prec, what=""):
  """CAM (nets/SqueezeSegV2.py:66-70) at its own output, float64 on the device's own 16-bit input (NHWC float32 GPU
  tensors), with the error the kernel's arithmetic allows.  U = 2^-11 (fp16) / 2^-8 (bf16):
    the 7x7 max is exact;
    squeeze: 16-bit weights, fp32 accumulation, the hidden vector s rounded to 16 bits:
      |ds| <= U (1.5 S1 + s), S1 = |W1| |pool| + |b1|; and ds = 0 where pre < -1.5 U S1 (the device's ReLU gives 0 too);
    excitation: 16-bit weights, b2 as a hi + lo pair of 16-bit values (float32 accurate):
      |de| <= (1 + U) |W2| ds + 1.5 U |W2| s + 2^-20 |b2|;
    gate: sigmoid's slope is <= 1/4; tanh.approx.f32 adds 0.5 |x| 2^-10; the output is rounded to 16 bits once.
  Near zero every 16-bit rounding is absolute (half the smallest subnormal)."""
  u, sub = U[prec], SUB[prec]
  k1, b1 = _fold64(p, name + "/squeeze", name + "/squeeze_bn")
  k2, b2 = _fold64(p, name + "/excitation", name + "/excitation_bn")
  x = x_dev.permute(0, 3, 1, 2).double()
  pool = O.max_pool_same(x, 7, (1, 1))
  pre = O.conv2d_same(pool, k1, b1)
  S1 = O.conv2d_same(pool.abs(), k1.abs(), b1.abs())
  s = torch.relu(pre)
  ds = torch.where(pre < -1.5 * u * S1, torch.zeros_like(s), u * (1.5 * S1 + s) + sub)
  del pool, S1
  e = O.conv2d_same(s, k2, b2)
  de = (1 + u) * O.conv2d_same(ds, k2.abs()) + 1.5 * u * O.conv2d_same(s, k2.abs()) + 2.0 ** -20 * b2.abs().view(1, -1, 1, 1)
  del s, ds, pre
  y = x * torch.sigmoid(e)
  bound = x.abs() * (0.25 * de + 0.5 * TANH) + u * y.abs() + sub
  got = y_dev.permute(0, 3, 1, 2).double()
  d = (got - y).abs()
  over = d > bound
  if bool(over.any()):
    r = d / bound
    i = np.unravel_index(int(r.argmax()), tuple(r.shape))
    raise AssertionError("%s: CAM error %.3g x the error model, %d elements over; worst at (b, c, h, w) = %s: got %r, "
                         "float64 %r, bound %.3g" % (what, float(r.max()), int(over.sum()), i, float(got[i]),
                                                     float(y[i]), float(bound[i])))
  return float((d / bound).max())


# ---- CAM cases ------------------------------------------------------------------------------------------------------
def _cam_case(cid, C, B, H, W, act="relu", mode=None, pool=False, bench=False):
  """mode: None | "zero-hidden" (squeeze BN beta -64: s = 0, the gate is sigmoid(b2)) | "saturated" (excitation BN
  beta +-12).  act None: c0 without activation (signed CAM input)."""
  return [pytest.param(dict(id=cid + "-" + prec, prec=prec, C=C, B=B, H=H, W=W, act=act, mode=mode, pool=pool,
                            bench=bench), id=cid + "-" + prec)
          for prec in PREC]


CAM_CASES = [
    # ---- the benchmark's CAM shapes and batches (KITTI 64x2048 and nuScenes 32x1024: CAM at W / 2), every frame ----
    *_cam_case("bench-kitti-c64-w1024-b32-pool", 64, 32, 64, 1024, pool=True, bench=True),
    *_cam_case("bench-kitti-c64-w1024-b1", 64, 1, 64, 1024, bench=True),
    *_cam_case("bench-kitti-c128-w512-b32", 128, 32, 64, 512, bench=True),
    *_cam_case("bench-kitti-c128-w512-b1-pool", 128, 1, 64, 512, pool=True, bench=True),
    *_cam_case("bench-nuscenes-c64-w512-b32", 64, 32, 32, 512, bench=True),
    *_cam_case("bench-nuscenes-c64-w512-b1", 64, 1, 32, 512, bench=True),
    *_cam_case("bench-nuscenes-c128-w256-b32-pool", 128, 32, 32, 256, pool=True, bench=True),
    *_cam_case("bench-nuscenes-c128-w256-b1", 128, 1, 32, 256, bench=True),
    # ---- segment plans (148 SMs): the comment gives segments x rows (+ the last segment's rows) ----
    *_cam_case("segs3-c64-h24-w100", 64, 1, 24, 100),                          # 3 x 8
    *_cam_case("segs3-short-last-c128-h64-w881-b2", 128, 2, 64, 881),          # 2 x 22 + 20
    *_cam_case("segs4-last-under-7-c64-h33-w40", 64, 1, 33, 40),               # 3 x 9 + 6
    *_cam_case("segs5-signed-c64-h40-w200", 64, 1, 40, 200, act=None),         # 5 x 8
    *_cam_case("segs5-signed-c128-h40-w130", 128, 1, 40, 130, act=None),       # 5 x 8
    *_cam_case("segs6-saturated-c64-h48-w100", 64, 1, 48, 100, mode="saturated"),
    *_cam_case("segs6-zero-hidden-c128-h48-w70", 128, 1, 48, 70, mode="zero-hidden"),
    *_cam_case("segs7-last-under-7-signed-c64-h64-w865-b2", 64, 2, 64, 865, act=None),   # 6 x 10 + 4
    *_cam_case("segs7-last-under-7-c128-h64-w881", 128, 1, 64, 881, pool=True),          # 6 x 10 + 4
    # ---- edges: the window taller than the image, narrower than the window, strip-width edges ----
    *_cam_case("edge-h1-c64-w70", 64, 3, 1, 70),
    *_cam_case("edge-h1-c128-w33-signed", 128, 2, 1, 33, act=None),
    *_cam_case("edge-h3-c128-w16-tw", 128, 4, 3, 16),
    *_cam_case("edge-h6-c64-w33-tw1-signed", 64, 2, 6, 33, act=None),
    *_cam_case("edge-w5-c64-h9", 64, 3, 9, 5, pool=True),
    *_cam_case("edge-w5-c128-h12-signed", 128, 2, 12, 5, act=None),
    *_cam_case("edge-w32-tw-c64-h12", 64, 2, 12, 32),
    *_cam_case("edge-w17-tw1-c128-h20", 128, 2, 20, 17),
    *_cam_case("c64-h11-w70-pool", 64, 2, 11, 70, pool=True),
    *_cam_case("c128-h11-w33-pool", 128, 2, 11, 33, pool=True),
    # ---- the gate's extremes ----
    *_cam_case("zero-hidden-c64-h16-w100", 64, 2, 16, 100, mode="zero-hidden"),
    *_cam_case("saturated-c128-h11-w33", 128, 2, 11, 33, mode="saturated"),
]


def _cam_cases():
  return [c.values[0] for c in CAM_CASES]


def test_cam_case_matrix():
  """At 148 SMs the CAM cases reach every segment count 1-8 for each C and precision, a last segment shorter than the
  others, a last segment shorter than the 7-row window, H < 7, signed input (also with several segments), both gate
  extremes and the benchmark's plans."""
  cases = _cam_cases()
  for C in (64, 128):
    for prec in PREC:
      cs = [c for c in cases if c["C"] == C and c["prec"] == prec]
      plans = [_cam_plan(C, c["B"], c["H"], c["W"], REF_SMS) for c in cs]
      assert {g[2] for g, _, _ in plans} == set(range(1, 9)), (C, prec, sorted({g[2] for g, _, _ in plans}))
      assert any(g[2] > 1 and last < rps for g, rps, last in plans), (C, prec)
      assert any(g[2] > 1 and last < 7 for g, _, last in plans), (C, prec)
      assert any(c["H"] < 7 for c in cs) and any(c["act"] is None for c in cs), (C, prec)
      assert any(c["act"] is None and p[0][2] > 1 for c, p in zip(cs, plans)), (C, prec)
      assert any(c["W"] % (256 // (C // 8)) for c in cs) and any(c["W"] < 7 for c in cs), (C, prec)
      assert any(c["W"] == 256 // (C // 8) for c in cs) and any(c["W"] == 256 // (C // 8) + 1 for c in cs), (C, prec)
      assert any(c["pool"] for c in cs) and {c["mode"] for c in cs} == {None, "zero-hidden", "saturated"}, (C, prec)
  bench = {(c["C"], c["H"], c["W"], c["B"], c["prec"]) for c in cases if c["bench"]}
  assert bench == {(C, H, W, B, p) for C, H, W in ((64, 64, 1024), (128, 64, 512), (64, 32, 512), (128, 32, 256))
                   for B in (32, 1) for p in PREC}


def _ncu_grids(path):
  rows = []
  with open(path) as f:
    lines = [ln for ln in f if not ln.startswith("==")]
  for r in csv.DictReader(lines):
    rows.append((r["Kernel Name"], tuple(int(v) for v in r["Grid Size"].strip("()").split(","))))
  return rows


def test_cam_and_input_plans_reproduce_the_recorded_grids():
  """The Python copies of launch_cam and launch_net_input give the grids Nsight Compute recorded for the benchmark
  (SqueezeSegV2 KITTI 64x2048, batch 32, fp16, 148 SMs; profiles/ncu_launches_r2.csv)."""
  rows = _ncu_grids(os.path.join(ROOT, "profiles", "ncu_launches_r2.csv"))
  cams = {}
  for name, grid in rows:
    inst = _cam_inst(name)
    if inst:
      cams.setdefault(inst[1], set()).add(grid)
    if "net_input_kernel" in name:
      assert grid == _input_grid(32 * 64 * 2048, REF_SMS), grid
  assert set(cams) == {64, 128}
  assert cams[64] == {_cam_plan(64, 32, 64, 1024, REF_SMS)[0]} == {(32, 32, 2)}
  assert cams[128] == {_cam_plan(128, 32, 64, 512, REF_SMS)[0]} == {(32, 32, 2)}


# ---- graphs ---------------------------------------------------------------------------------------------------------
def _c0(g, C, act):
  y = L.BatchNormalization("c0_bn")(L.Conv2D("c0", C, 3)(g.input))
  return L.relu(y) if act == "relu" else y


class _Net:
  def __init__(self, t, prec, B, opts):
    self.t, self.lib, self.B = t, _lib.load(), B
    o = {"use_graph": 0, "keep_tensors": 1, "micro_batch": 0}
    o.update(opts)
    self.h = t.g.build_net(t.logits, 2, 0, PREC[prec], B, o)
    mb = o["micro_batch"]
    self.passes = -(-B // mb) if mb else 1
    self.last = B - (self.passes - 1) * mb if mb else B

  def forward(self, x):
    xd = torch.from_numpy(x).cuda()
    preds = torch.empty(x.shape[:3], dtype=torch.int32, device="cuda")
    _lib.check(self.lib.pcls_net_forward(self.h, xd.data_ptr(), 6, None, None, None, x.shape[0], None, None,
                                         preds.data_ptr(), torch.cuda.current_stream().cuda_stream), "pcls_net_forward")
    torch.cuda.synchronize()

  def read(self, sym):
    """The last pass's frames of `sym` as float32 NHWC on the GPU."""
    o = torch.empty((self.last, self.t.g.H, sym.width, sym.channels), dtype=torch.float32, device="cuda")
    _lib.check(self.lib.pcls_net_read_tensor(self.h, sym.tid, self.last, o.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "pcls_net_read_tensor")
    torch.cuda.synchronize()
    return o

  def close(self):
    self.lib.pcls_net_destroy(self.h)


class CamCase:
  def __init__(self, c):
    self.c = c
    self.t = TinyNet(c["H"], c["W"])
    g = self.t.g
    self.inp = _c0(g, c["C"], c["act"])
    self.cam = g.cam(self.inp, "cam", c["C"] // 16)
    self.out = L.max_pool2d(self.cam) if c["pool"] else self.cam
    self.rng = np.random.default_rng(zlib.crc32(c["id"].encode()))
    _rand_vars(g, self.rng)
    if c["mode"] == "zero-hidden":
      g.variables["cam/squeeze_bn/beta"][:] = -64.0
    elif c["mode"] == "saturated":
      beta = g.variables["cam/excitation_bn/beta"]
      beta[:] = np.where(np.arange(beta.size) % 2 == 0, 12.0, -12.0)
    self.p = {k: v.cuda() for k, v in _tp(g).items()}

  def net(self, B=None, **opts):
    return _Net(self.t, self.c["prec"], B or self.c["B"], opts)


def _check_cam_values(case, inp, out, what):
  """Check 1 in frame chunks (bounded float64 memory)."""
  c = case.c
  step = max(1, (1 << 25) // (c["H"] * c["W"] * c["C"]))
  for f0 in range(0, inp.shape[0], step):
    _check_cam(inp[f0:f0 + step], out[f0:f0 + step], case.p, "cam", c["prec"], "%s, frames %d.." % (what, f0))


@pytest.mark.gpu
@pytest.mark.parametrize("c", CAM_CASES)
def test_cam_against_float64(c):
  case = CamCase(c)
  B, H, W, C, prec = c["B"], c["H"], c["W"], c["C"], c["prec"]
  sms = _sms()
  x1, x2 = _input(case.rng, B, H, W), _input(case.rng, B, H, W)
  main = case.net()
  try:
    # ---- check 4: kernel, launch count, grid ----
    trace = _trace(lambda: main.forward(x1))
    _check_launches(main.lib, main.h, 1, trace)
    cams = [(n, gr) for n, gr in trace if _cam_inst(n)]
    assert len(cams) == 1, trace
    assert _cam_inst(cams[0][0]) == (TNAME[prec], C), "the CAM ran %s" % cams[0][0]
    assert cams[0][1] == _cam_plan(C, B, H, W, sms)[0], "grid %s, launch_cam plans %s at %d SMs" % (
        cams[0][1], _cam_plan(C, B, H, W, sms)[0], sms)
    if c["pool"]:
      pools = [(n, gr) for n, gr in trace if _tmpl(n, "maxpool3x3_s2_kernel")]
      assert len(pools) == 1 and _tmpl(pools[0][0], "maxpool3x3_s2_kernel") == TNAME[prec], trace
      assert pools[0][1] == _pool_plan(C, B, H, W, sms)[0], pools

    # ---- checks 1 and 2: the second forward, every pixel of every frame ----
    main.forward(x2)
    inp, cam = main.read(case.inp), main.read(case.cam)
    _check_cam_values(case, inp, cam, "C %d B %d H %d W %d %s" % (C, B, H, W, prec))
    out = cam
    if c["pool"]:
      out = main.read(case.out)
      ref = O.max_pool_same(cam.permute(0, 3, 1, 2), 3, (1, 2)).permute(0, 2, 3, 1)
      assert torch.equal(out, ref), "the max-pool behind the CAM is not the exact max-pool of its input"
    del inp, cam

    # ---- check 3: other plumbing ----
    main.forward(x2)
    assert torch.equal(main.read(case.out), out), "a repeated forward is not bit-identical"
    net = case.net(keep_tensors=0, use_graph=1)
    try:
      for i in range(3):                                                   # capture, then replays
        net.forward(x2)
        assert torch.equal(net.read(case.out), out), "keep_tensors = 0, use_graph = 1, call %d: outputs differ" % i
    finally:
      net.close()
    if B > 1:                                                              # one frame per pass: another plan
      net = case.net(micro_batch=1)
      xs, want = x2, out[-1:]
    else:                                                                  # three copies of the frame
      net = case.net(B=3)
      xs, want = np.repeat(x2, 3, 0), out.expand(3, -1, -1, -1)
    try:
      net.forward(xs)
      assert torch.equal(net.read(case.out), want), "another row-segment plan (%s vs %s) gives other bits" % (
          _cam_plan(C, net.last, H, W, sms)[0], _cam_plan(C, B, H, W, sms)[0])
    finally:
      net.close()
  finally:
    main.close()


# ---- max-pool -------------------------------------------------------------------------------------------------------
def _pool_case(cid, C, B, H, W, act=None):
  return [pytest.param(dict(id=cid + "-" + prec, prec=prec, C=C, B=B, H=H, W=W, act=act), id=cid + "-" + prec)
          for prec in PREC]


POOL_CASES = [
    *_pool_case("even-w130-c64-h64-signed", 64, 2, 64, 130),          # pad_left 0, 8 segments x 8
    *_pool_case("odd-w129-c128-h60-signed", 128, 2, 60, 129),         # pad_left 1, 6 x 9 + 6
    *_pool_case("odd-w257-c64-h5-b3", 64, 3, 5, 257, act="relu"),     # one segment
    *_pool_case("odd-w3-c32-h20-signed", 32, 2, 20, 3),               # Wout 2, 2 x 10
    *_pool_case("even-w1024-c64-h64-b32-signed", 64, 32, 64, 1024),   # the benchmark's pool1 input: 4 x 13 + 12
]


def test_pool_case_matrix():
  for prec in PREC:
    cs = [c.values[0] for c in POOL_CASES if c.values[0]["prec"] == prec]
    plans = [_pool_plan(c["C"], c["B"], c["H"], c["W"], REF_SMS) for c in cs]
    assert any(c["W"] % 2 == 0 for c in cs) and any(c["W"] % 2 for c in cs)
    assert any(c["act"] is None and c["W"] % 2 for c in cs) and any(c["act"] is None and c["W"] % 2 == 0 for c in cs)
    assert any(g[1] > 2 for g, _, _ in plans) and any(g[1] > 1 and last < rps for g, rps, last in plans)


@pytest.mark.gpu
@pytest.mark.parametrize("fused_off", [False, True], ids=["last-op", "fuse_pool0"])
@pytest.mark.parametrize("c", POOL_CASES)
def test_maxpool_exact(c, fused_off):
  """maxpool3x3_s2_kernel against O.max_pool_same on the device's own input, as the graph's last op (conv_impl = 0)
  and in front of a 1x1 conv with fuse_pool = 0."""
  B, H, W, C, prec = c["B"], c["H"], c["W"], c["C"], c["prec"]
  t = TinyNet(H, W)
  g = t.g
  a = _c0(g, C, c["act"])
  pooled = L.max_pool2d(a)
  if fused_off:
    L.relu(L.Conv2D("sq", 16, 1)(pooled))
  rng = np.random.default_rng(zlib.crc32(c["id"].encode()))
  _rand_vars(g, rng)
  x1, x2 = _input(rng, B, H, W), _input(rng, B, H, W)
  opts = {"conv_impl": 0, "fuse_pool": 0} if fused_off else {"conv_impl": 0}
  net = _Net(t, prec, B, opts)
  try:
    trace = _trace(lambda: net.forward(x1))
    _check_launches(net.lib, net.h, 1, trace)
    pools = [(n, gr) for n, gr in trace if _tmpl(n, "maxpool3x3_s2_kernel")]
    assert len(pools) == 1 and _tmpl(pools[0][0], "maxpool3x3_s2_kernel") == TNAME[prec], trace
    assert pools[0][1] == _pool_plan(C, B, H, W, _sms())[0], pools
    net.forward(x2)                                                       # the second forward is checked
    ya, yp = net.read(a), net.read(pooled)
    ref = O.max_pool_same(ya.permute(0, 3, 1, 2), 3, (1, 2)).permute(0, 2, 3, 1)
    assert torch.equal(yp, ref), "max-pool differs from the exact max at %d elements" % int((yp != ref).sum())
    if c["act"] is None:
      assert bool((ya < 0).any()) and bool((yp < 0).any())               # signed: only -inf padding is right
  finally:
    net.close()
  g2 = _Net(t, prec, B, dict(opts, keep_tensors=0, use_graph=1))
  try:
    for i in range(2):
      g2.forward(x2)
      assert torch.equal(g2.read(pooled), yp), "keep_tensors = 0, use_graph = 1, call %d: outputs differ" % i
  finally:
    g2.close()


# ---- network input --------------------------------------------------------------------------------------------------
MEAN5 = (10.88, 0.23, -1.04, 0.21, 12.12)
STD5 = (11.47, 6.91, 0.86, 0.16, 12.32)


def _dptr(vals):
  return (ctypes.c_double * 5)(*vals)


class _InputNet:
  """TinyNet's throw-away logits conv of the input: the forward is the input kernel, the 1x1 logits conv and the head."""

  def __init__(self, prec, B, H, W, seed=5):
    self.prec, self.B, self.H, self.W = prec, B, H, W
    self.t = TinyNet(H, W)
    _rand_vars(self.t.g, np.random.default_rng(seed))
    self.lib = _lib.load()
    self.h = self.t.g.build_net(self.t.logits, 2, 0, PREC[prec], B, {"use_graph": 0})

  def run(self, x, channels, mask=None, raw=False, in16=False):
    """x: torch CPU tensor [B,H,W,channels] (float32, or the 16-bit storage type with in16).  Returns (tensor 0 bits,
    mask buffer, predictions) on the GPU."""
    xd = x.contiguous().cuda()
    md = None if mask is None else torch.as_tensor(mask, dtype=torch.uint8).contiguous().cuda()
    preds = torch.empty((self.B, self.H, self.W), dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    mp = None if md is None else md.data_ptr()
    if in16:
      _lib.check(self.lib.pcls_net_forward_in16(self.h, xd.data_ptr(), channels, mp, self.B, None, None,
                                                preds.data_ptr(), st), "pcls_net_forward_in16")
    else:
      mean, std = (_dptr(MEAN5), _dptr(STD5)) if raw else (None, None)
      _lib.check(self.lib.pcls_net_forward(self.h, xd.data_ptr(), channels, mp, mean, std, self.B, None, None,
                                           preds.data_ptr(), st), "pcls_net_forward")
    torch.cuda.synchronize()
    t0, m = _input_buffers(self.lib, self.h, self.B, self.H, self.W)
    rd = torch.empty((self.B, self.H, self.W, 8), dtype=torch.float32, device="cuda")
    _lib.check(self.lib.pcls_net_read_tensor(self.h, 0, self.B, rd.data_ptr(), st), "pcls_net_read_tensor")
    torch.cuda.synchronize()
    assert bool(_same16(rd.to(DT[self.prec]).view(torch.int16), t0, self.prec).all()), "read_tensor(0) differs"
    return t0, m, preds

  def close(self):
    self.lib.pcls_net_destroy(self.h)


def _ref_normalised(x6, prec):
  """Tensor 0 of a normalised float32 input: channels 0-5 rounded to T, pads 6-7 = +0."""
  b = _bits(x6, prec)
  return torch.cat([b, torch.zeros(b.shape[:3] + (2,), dtype=torch.int16)], -1)


def _nonzero16(bits):
  return (bits & 0x7FFF) != 0


def _assert_input(t0, m, ref_t0, ref_m, prec, what):
  ref_t0, ref_m = ref_t0.cuda(), ref_m.cuda().to(torch.uint8)
  bad = ~_same16(t0, ref_t0, prec)
  assert not bool(bad.any()), "%s: tensor 0 differs at %d elements, first at %s" % (
      what, int(bad.sum()), tuple(int(v) for v in bad.nonzero()[0]))
  assert torch.equal(m, ref_m), "%s: mask differs at %d pixels" % (what, int((m != ref_m).sum()))


def _signed_input(rng, B, H, W):
  x = torch.from_numpy(rng.normal(0, 3, (B, H, W, 6)).astype(np.float32))
  ch5 = rng.choice(np.array([0.0, 1.0, 1.0, -0.0, 0.3, -2.0], np.float32), (B, H, W))
  x[..., 5] = torch.from_numpy(ch5)
  return x


@pytest.mark.gpu
@pytest.mark.parametrize("with_mask", [False, True], ids=["derived-mask", "given-mask"])
@pytest.mark.parametrize("prec", list(PREC))
def test_net_input_normalised_f32_bit_exact(prec, with_mask):
  B, H, W = 2, 16, 100
  rng = np.random.default_rng(21)
  x = _signed_input(rng, B, H, W)
  mask = torch.from_numpy(rng.choice(np.array([0, 1, 7, 255], np.uint8), (B, H, W))) if with_mask else None
  net = _InputNet(prec, B, H, W)
  try:
    t0, m, _ = net.run(x, 6, mask)
  finally:
    net.close()
  ref = _ref_normalised(x, prec)
  ref_m = (mask != 0) if with_mask else _nonzero16(ref[..., 5])
  _assert_input(t0, m, ref, ref_m, prec, "normalised f32 %s" % prec)


def _raw_input(rng, B, H, W, channels):
  x = torch.from_numpy(rng.normal(0, 20, (B, H, W, channels)).astype(np.float32))
  depth = rng.choice(np.array([np.nan, -0.0, 0.0, -3.0, 1e-30, 7.5, 40.0, 80.0, np.inf], np.float32), (B, H, W))
  x[..., 4] = torch.from_numpy(depth)
  return x


@pytest.mark.gpu
@pytest.mark.parametrize("with_mask", [False, True], ids=["derived-mask", "given-mask"])
@pytest.mark.parametrize("channels", [5, 6])
@pytest.mark.parametrize("prec", list(PREC))
def test_net_input_raw_bit_exact(prec, channels, with_mask):
  """Raw x, y, z, i, d (, label) with the input stage fused: m = depth > 0 (NaN, -0, 0 and negative depths are empty),
  T(float32((float64(x) - mean) / std)) where m holds and 0 elsewhere, channel 5 = m.  A given mask sets the mask
  buffer only; channel 5 still follows the depth."""
  B, H, W = 2, 16, 100
  rng = np.random.default_rng(22 + channels)
  x = _raw_input(rng, B, H, W, channels)
  mask = torch.from_numpy(rng.integers(0, 2, (B, H, W)).astype(np.uint8)) if with_mask else None
  net = _InputNet(prec, B, H, W)
  try:
    t0, m, _ = net.run(x, channels, mask, raw=True)
  finally:
    net.close()
  x64 = x[..., :5].double()
  valid = x64[..., 4] > 0
  norm = ((x64 - torch.tensor(MEAN5, dtype=torch.float64)) / torch.tensor(STD5, dtype=torch.float64)).float()
  norm = torch.where(valid[..., None], norm, torch.zeros_like(norm))
  ref = _ref_normalised(torch.cat([norm, valid[..., None].float()], -1), prec)
  _assert_input(t0, m, ref, (mask != 0) if with_mask else valid, prec, "raw %d channels %s" % (channels, prec))


@pytest.mark.gpu
@pytest.mark.parametrize("with_mask", [False, True], ids=["derived-mask", "given-mask"])
@pytest.mark.parametrize("channels", [6, 8])
@pytest.mark.parametrize("prec", list(PREC))
def test_net_input16_bit_exact(prec, channels, with_mask):
  """A pure re-pack of arbitrary 16-bit patterns (NaN payloads included): channels 0-5 as given, pads 6-7 zero even
  when the input's are not; the derived mask is channel 5 != +-0 (NaN is valid)."""
  B, H, W = 2, 16, 100
  rng = np.random.default_rng(23 + channels)
  bits = torch.from_numpy(rng.integers(-32768, 32768, (B, H, W, channels)).astype(np.int16))
  bits[0, :, :8, 5] = torch.tensor([0, -32768, 0x7E00, -1, 1, 0x7C00, 0x3C00, 0], dtype=torch.int16)  # +0 -0 NaN ...
  bits[1, :, :4, 5] = 0
  mask = torch.from_numpy(rng.integers(0, 2, (B, H, W)).astype(np.uint8)) if with_mask else None
  net = _InputNet(prec, B, H, W)
  try:
    t0, m, _ = net.run(bits.view(DT[prec]), channels, mask, in16=True)
  finally:
    net.close()
  ref = torch.cat([bits[..., :6], torch.zeros((B, H, W, 2), dtype=torch.int16)], -1)
  assert torch.equal(t0, ref.cuda()), "tensor 0 is not the bit-exact re-pack"
  ref_m = (mask != 0) if with_mask else _nonzero16(bits[..., 5])
  assert torch.equal(m, ref_m.cuda().to(torch.uint8)), "mask differs at %d pixels" % int((m.cpu() != ref_m).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("prec", list(PREC))
def test_net_input_above_the_grid_cap(prec):
  """The benchmark's 32 x 64 x 2048 pixels: several trips through the grid-stride loop of both input kernels."""
  B, H, W = 32, 64, 2048
  n = B * H * W
  grid = _input_grid(n, _sms())
  assert n > 2 * grid[0] * 256
  rng = np.random.default_rng(24)
  x = _signed_input(rng, B, H, W)
  ref = _ref_normalised(x, prec)
  ref_m = _nonzero16(ref[..., 5])
  net = _InputNet(prec, B, H, W)
  try:
    trace = _trace(lambda: net.run(x, 6))
    ins = [(nm, gr) for nm, gr in trace if "net_input" in nm]
    assert len(ins) == 1 and _tmpl(ins[0][0], "net_input_kernel") == TNAME[prec] and ins[0][1] == grid, ins
    t0, m, _ = net.run(x, 6)
    _assert_input(t0, m, ref, ref_m, prec, "f32 entry point, %d pixels" % n)
    x16 = x.to(DT[prec])
    trace = _trace(lambda: net.run(x16, 6, in16=True))
    ins = [(nm, gr) for nm, gr in trace if "net_input" in nm]
    assert len(ins) == 1 and "net_input16_kernel" in ins[0][0] and ins[0][1] == grid, ins
    t0, m, _ = net.run(x16, 6, in16=True)
    _assert_input(t0, m, ref, ref_m, prec, "16-bit entry point, %d pixels" % n)
  finally:
    net.close()


MASK_EDGES = np.array([0.0, -0.0, np.nan, np.inf, -np.inf, 1e-8, -1e-8, 2.9e-8, 6e-8, 1e-40, -1e-40, 1.4e-45, 1e-39,
                       1.0, 0.5, -1.0], np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("prec", list(PREC))
def test_mask_channel_edges_agree_across_entry_points(prec):
  """mask = NULL: both entry points derive the mask from channel 5 as tensor 0 stores it (T(ch5) != +-0), so a float32
  channel 5 that rounds to a 16-bit zero (1e-8 in fp16, 1.4e-45 in both) is invalid through either, like NaN is valid.
  Tensor 0, the mask and the predictions agree pixel by pixel."""
  B, H, W = 2, 8, 64
  rng = np.random.default_rng(25)
  x = torch.from_numpy(rng.normal(0, 1, (B, H, W, 6)).astype(np.float32))
  x[..., 5] = torch.from_numpy(MASK_EDGES[rng.integers(0, MASK_EDGES.size, (B, H, W))])
  x[0, 0, :MASK_EDGES.size, 5] = torch.from_numpy(MASK_EDGES)
  ref = _ref_normalised(x, prec)
  ref_m = _nonzero16(ref[..., 5])
  if prec == "f16":
    assert not bool(ref_m[0, 0, 5]) and bool(x[0, 0, 5, 5] != 0)       # 1e-8: a float32 nonzero, an fp16 zero
  net = _InputNet(prec, B, H, W)
  try:
    t32, m32, p32 = net.run(x, 6)
    t16, m16, p16 = net.run(x.to(DT[prec]), 6, in16=True)
  finally:
    net.close()
  _assert_input(t32, m32, ref, ref_m, prec, "f32 entry point")
  _assert_input(t16, m16, ref, ref_m, prec, "16-bit entry point")
  assert torch.equal(p32, p16), "predictions differ at %d pixels" % int((p32 != p16).sum())
  assert bool((p32[~ref_m.cuda()] == 0).all())                          # none_index where the mask is 0


# ---- census of the benchmarked networks -----------------------------------------------------------------------------
def _owned(prec):
  """{kernel family: set of template arguments (or None)} that a per-op test declares for precision `prec`."""
  own = {"cam2_kernel": {c["C"] for c in _cam_cases() if c["prec"] == prec},
         "maxpool3x3_s2_kernel": {None} if any(c.values[0]["prec"] == prec for c in POOL_CASES) else set(),
         "net_input_kernel": {None}, "net_input16_kernel": {None},
         "head_kernel": {None} if any(c.values[0]["path"] in ("C", "D") for c in LH.CASES) else set(),
         "conv_head_kernel": {c.values[0]["inst"] for c in LH.CASES if c.values[0]["path"] == "A"
                              and c.values[0]["prec"] == prec}}
  for fam, k in CK.FAMILY.items():
    own[k] = {tuple(i[1:]) for i, p in CK._declared(("wrap", "bench", None)) if p == prec and i[0] == fam}
  return own


def _family(name):
  """(family, template arguments after T or None) of a pcls:: kernel name; None for kernels outside the project."""
  if "pcls::" not in name and "4pcls" not in name:
    return None
  inst = CK._inst(name)
  if inst is not None:
    return CK.FAMILY[inst[0]], inst[2]
  if "conv_head_kernel" in name:
    kc, cs, _ = LH._head_inst(name)
    return "conv_head_kernel", (kc, cs)
  ci = _cam_inst(name)
  if ci is not None:
    return "cam2_kernel", ci[1]
  m = re.search(r"(\w+_kernel)", name)
  return (m.group(1) if m else name), None


@pytest.mark.gpu
@pytest.mark.parametrize("prec", list(PREC))
@pytest.mark.parametrize("net", CK._bench_networks(), ids=lambda n: "%s-%s-%dx%d" % n)
def test_census_every_forward_kernel_has_a_per_op_test(net, prec):
  """Each pcls:: kernel a benchmarked network's forward launches (B = 1) is owned by a per-op test, and for SqueezeSegV2
  each CAM's shape and segment plan, at the benchmark batch and at B = 1, is one of this file's benchmark cases."""
  import bench
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
  names = CK._profiled(lambda: model.forward_device(x))
  model._release()
  fams = [f for f in (_family(n) for n in names) if f is not None]
  assert any(f[0] == "net_input_kernel" for f in fams), names
  own = _owned(prec)
  orphans = sorted({f for f in fams if f[1] not in own.get(f[0], ())}, key=str)
  assert not orphans, "%s %s launches kernels no per-op test owns: %s" % (name, prec, orphans)
  other = "__half" if prec == "bf16" else "__nv_bfloat16"
  assert not [n for n in names if "pcls::" in n and other in n], names
  cams = [op for op in model._graph.program if op["op"] == "cam"]
  assert bool(cams) == (name == "squeezesegv2")
  batch = {m_[:4]: m_[4] for m_ in bench.WORKLOADS.values()}[net]
  sms = _sms()
  declared = {(c["C"], c["H"], c["W"], c["B"], _cam_plan(c["C"], c["B"], c["H"], c["W"], sms)[0])
              for c in _cam_cases() if c["bench"] and c["prec"] == prec}
  for op in cams:
    C, Wc = op["channels"], op["src"].width
    for B in (batch, 1):
      key = (C, H, Wc, B, _cam_plan(C, B, H, Wc, sms)[0])
      assert key in declared, "%s: CAM %s (C, H, W, B, grid) = %s is not a benchmark case here" % (name, op["name"], key)
