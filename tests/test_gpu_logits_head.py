"""The logits layer and the segmentation head (softmax -> argmax -> mask, nets/SegmentationNetwork.py:58-69) against a
float64 reference, on every kernel that runs them:

  A  conv_head_kernel<T, KC, CS>: 3x3 logits conv with the head fused (or logits only with fuse_head = 0)
  B  conv_tc_kernel, float32 epilogue with the head fused (W % 128 == 0, the layer does not qualify for A)
  C  conv_tc_kernel writes the logits, then the standalone head_kernel (W % 128 != 0, or fuse_head = 0)
  D  conv_direct_kernel + head_kernel (conv_impl = 1)

Each case is a two-layer net built with nets/layers.Graph: input -> c0 (3x3 conv to Cin channels, BN, ReLU) -> head
(Conv2D(NC, k) with bias and BN: the net's logits).  c0's output is read back with keep_tensors = 1, so the reference
runs on the exact 16-bit values the logits layer consumed.  The forward gets an explicit mask array that differs from
input channel 5, and logits / probs / preds buffers with guard bands (interior prefilled with NaN / -7, guards with a
sentinel).  Every case checks:

  1. logits against float64 on the device's own input: |d| <= U * 1.5 * S + eps, U = 2^-11 (fp16) / 2^-8 (bf16),
     S = sum |w'| |x| (+ |b'|) - weight rounding plus fp32 accumulation; the float32 logits are not rounded again;
  2. probabilities against a float64 softmax of the device's own logits, with the bound of _softmax_bound (derived
     from the instructions of the kernel that computed them); finite, rows sum to 1, no mass on padding classes;
  3. predictions, exactly, on every in-image pixel: argmax of the device's probabilities (first index on ties) where
     the mask is 1, none_index where it is 0; the oracle's label wherever its top-2 margin exceeds twice the logit bound;
  4. nothing written outside [B,H,W,NC], nothing left unwritten inside;
  5. the same answer through other plumbing: logits = probs = NULL, keep_tensors = 0, fuse_head = 0 (bit-identical
     logits; labels equal unless the two best logits are within the rounding of the two softmax implementations);
  6. the kernel sequence of one forward (torch.profiler, CUDA activity) names the path the case claims, and
     pcls_net_launches_per_forward agrees with it.  A planner change that moves a case to another path fails here.
"""
import math
import re
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import nn as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.nets import layers as L

pytestmark = pytest.mark.gpu

HD_TILE = 126                  # output pixels per conv_head_kernel tile (conv_head.cu)
HD_NG = 4                      # epilogue groups per conv_head_kernel CTA
GUARD = 256                    # guard elements on each side of every output buffer (1 KB keeps 16-byte alignment)
F_SENT = np.float32(-1.25e37)  # guard sentinels
I_SENT = 0x5A5A5A5A
U16 = {"f16": 2.0 ** -11, "bf16": 2.0 ** -8}
PREC = {"f16": _lib.PCLS_F16, "bf16": _lib.PCLS_BF16}
LOG2E = 1.0 / math.log(2.0)
u = 2.0 ** -24                 # float32 unit roundoff

# Per kernel: (k_a, k_m, e_exp, e_div) for the softmax error model of _softmax_bound.
#   conv_head_kernel  a = fma(l, L2E, -mx * L2E) - L2E = fl32(log2 e), the product mx * L2E and the fma each round once:
#                     |da| <= u log2e (2 |l - mx| + |mx|)  (the |mx| term is the rounding of mx * L2E: it grows with the
#                     largest logit);  ex2.approx.ftz (PTX ISA: 2 ulp; allowed 4 ulp = 2^-21), fp32 sum,
#                     __fdividef(1, sum) (2 ulp) and the product with it (1 rounding): 2^-22 + 2^-24
#   conv_tc_kernel    a = (l - mx) * L2E: the difference, L2E and the product: |da| <= 3 u log2e |l - mx|;
#                     ex2.approx.ftz, fp32 sum, __fdividef and the product as above
#   head_kernel       expf(l - mx) (2 ulp = 2^-22 on top of the rounding of l - mx: |da| <= u log2e |l - mx|),
#                     fp32 sum, __fdiv_rn (correctly rounded: 2^-24)
SOFTMAX_ERR = {"conv_head": (2.0, 1.0, 2.0 ** -21, 2.0 ** -22 + u),
               "conv_tc": (3.0, 0.0, 2.0 ** -21, 2.0 ** -22 + u),
               "head": (1.0, 0.0, 2.0 ** -22, u)}
KERNEL_RE = re.compile(r"(net_input\w*|conv_\w+|head)_kernel")   # the kernels a forward of these nets launches
PATH_KERNEL = {"A": "conv_head_kernel", "B": "conv_tc_kernel", "C": "conv_tc_kernel", "D": "conv_direct_kernel"}


def _case(cid, cin, nc, H, W, B, path, prec="f16", k=3, act=None, impl=0, mb=0, none="0", weights="rand", inst=None,
          regime=None):
  """inst = (KC, CS) of the conv_head_kernel instantiation a path-A case must run; regime = the tile regime it claims."""
  return pytest.param(dict(cin=cin, nc=nc, H=H, W=W, B=B, path=path, prec=prec, k=k, act=act, impl=impl, mb=mb,
                           none=none, weights=weights, inst=inst, regime=regime), id=cid)


CASES = [
    # ---- path A: all 16 instantiations (KC 32 / 64 x CS 8 / 12 / 16 / 20 x fp16 / bf16), cout % 4 == 0 and != 0 ----
    _case("A-kc32-cs8-f16-nc5-w100", 32, 5, 5, 100, 2, "A", inst=(32, 8), regime="few"),
    _case("A-kc32-cs12-f16-nc12-w252-h2", 32, 12, 2, 252, 3, "A", none="last", inst=(32, 12), regime="few"),
    _case("A-kc32-cs16-f16-nc13-w253-h1", 32, 13, 1, 253, 2, "A", inst=(32, 16), regime="few"),
    _case("A-kc32-cs20-f16-nc20-w127", 32, 20, 5, 127, 2, "A", inst=(32, 20), regime="few"),
    _case("A-kc64-cs8-f16-nc8-w128-leaky", 64, 8, 2, 128, 2, "A", act="leaky", inst=(64, 8)),
    _case("A-kc64-cs12-f16-nc11-w126-relu", 64, 11, 5, 126, 2, "A", act="relu", inst=(64, 12)),
    _case("A-kc64-cs16-f16-nc16-w64", 64, 16, 6, 64, 3, "A", none="last", inst=(64, 16)),
    _case("A-kc64-cs20-f16-nc19-S2-1to4-per-cta", 64, 19, 16, 253, 10, "A", inst=(64, 20), regime="1-4"),
    _case("A-kc64-cs20-f16-nc20-S3-64x2048-b4-wrap", 64, 20, 64, 2048, 4, "A", inst=(64, 20), regime="wrap-in-frame"),
    _case("A-kc32-cs8-bf16-nc8-w64-h2", 32, 8, 2, 64, 2, "A", prec="bf16", inst=(32, 8)),
    _case("A-kc32-cs12-bf16-nc11-w253", 32, 11, 5, 253, 2, "A", prec="bf16", none="last", inst=(32, 12)),
    _case("A-kc32-cs16-bf16-nc16-w127-h1", 32, 16, 1, 127, 3, "A", prec="bf16", inst=(32, 16)),
    _case("A-kc32-cs20-bf16-nc19-4x253-b300-wrap", 32, 19, 4, 253, 300, "A", prec="bf16", inst=(32, 20),
          regime="wrap-frames"),
    _case("A-kc64-cs8-bf16-nc5-w100", 64, 5, 5, 100, 2, "A", prec="bf16", inst=(64, 8)),
    _case("A-kc64-cs12-bf16-nc12-w252-leaky", 64, 12, 2, 252, 2, "A", prec="bf16", act="leaky", inst=(64, 12)),
    _case("A-kc64-cs16-bf16-nc13-w128", 64, 13, 5, 128, 2, "A", prec="bf16", inst=(64, 16)),
    _case("A-kc64-cs20-bf16-nc20-w126", 64, 20, 6, 126, 2, "A", prec="bf16", inst=(64, 20)),
    # ---- stage-count boundaries of head_plan_layer (Cin 96: S = 2 at NC 20, < 2 at NC 19; Cin 128: 1 stage) ----
    _case("A-cin96-nc20-S2", 96, 20, 3, 253, 2, "A", inst=(32, 20)),
    _case("B-cin96-nc19-1stage", 96, 19, 3, 256, 2, "B"),
    _case("B-cin128-nc20-1stage", 128, 20, 3, 256, 2, "B"),
    _case("A-cin48-padded-to-64", 48, 20, 3, 128, 2, "A", inst=(64, 20)),
    # ---- paths B / C / D ----
    _case("B-nc21-w256", 64, 21, 3, 256, 2, "B"),
    _case("B-nc32-w256", 64, 32, 3, 256, 2, "B", none="last"),
    _case("C-nc21-w250", 64, 21, 3, 250, 2, "C"),
    _case("C-nc32-w250", 64, 32, 3, 250, 2, "C", none="last"),
    _case("B-1x1-cout16-tmem_ld16", 64, 13, 3, 256, 2, "B", k=1),
    _case("C-w63", 64, 20, 3, 63, 2, "C"),
    _case("B-bf16-nc21-leaky", 64, 21, 3, 256, 2, "B", prec="bf16", act="leaky"),
    _case("B-nc24-relu", 64, 24, 3, 256, 2, "B", act="relu"),
    _case("D-conv_impl1", 64, 20, 3, 100, 2, "D", impl=1),
    # ---- semantics ----
    _case("A-ties-duplicated-classes", 64, 11, 5, 252, 2, "A", weights="ties", inst=(64, 12)),
    _case("B-ties-duplicated-classes", 64, 21, 3, 256, 2, "B", weights="ties"),
    _case("A-zero-weights-equal-bias", 32, 13, 3, 128, 2, "A", weights="zero", none="last", inst=(32, 16)),
    _case("B-zero-weights-equal-bias", 64, 24, 3, 256, 2, "B", weights="zero", none="last"),
    _case("A-large-logits", 64, 20, 5, 253, 2, "A", weights="large", inst=(64, 20)),
    _case("B-large-logits", 64, 21, 3, 256, 2, "B", weights="large"),
    _case("A-micro_batch3-b7", 64, 19, 5, 253, 7, "A", mb=3, none="last", inst=(64, 20)),
]


def test_case_matrix_covers_every_conv_head_instantiation():
  got = {(c.values[0]["inst"], c.values[0]["prec"]) for c in CASES if c.values[0]["path"] == "A"}
  want = {((kc, cs), p) for kc in (32, 64) for cs in (8, 12, 16, 20) for p in ("f16", "bf16")}
  assert want <= got, sorted(want - got)


# ---- helpers -----------------------------------------------------------------------------------------------------
def _f16(a):
  return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


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


TIE_PAIRS = ((1, 5), (2, 9))   # class j gets class i's kernel, bias and BN: bit-identical logits, the lower index must win


def _head_weights(g, mode):
  v = g.variables
  hk, hb = "head/kernel", "head/bias"
  bn = ["bh/gamma", "bh/beta", "bh/moving_mean", "bh/moving_variance"]
  if mode == "ties":
    for n, (i, j) in enumerate(TIE_PAIRS):
      v["bh/beta"][i] += 6.0 - 2.0 * n   # (after BN's scale) both duplicated pairs win on many pixels
      v[hk][..., j] = v[hk][..., i]
      for n in [hb] + bn:
        v[n][j] = v[n][i]
  elif mode == "zero":
    v[hk][...] = 0.0
    v[hb][...] = 0.3
    for n, val in zip(bn, (1.1, 0.2, 0.1, 0.9)):
      v[n][...] = val
  elif mode == "large":
    v[hk] *= 400.0
    v[hb] *= 400.0


def _fold64(p, conv, bn):
  k = p[conv + "/kernel"].double()
  b = p[conv + "/bias"].double()
  sc = p[bn + "/gamma"].double() / torch.sqrt(p[bn + "/moving_variance"].double() + O.BN_EPS)
  return k * sc.view(1, 1, 1, -1), (b - p[bn + "/moving_mean"].double()) * sc + p[bn + "/beta"].double()


def _conv_same_rows(x, k, b, rows=16):
  """O.conv2d_same, evaluated a band of output rows at a time (bounds the float64 im2col buffer at 64 x 2048)."""
  kh, kw = k.shape[0], k.shape[1]
  pt, pb = O.same_pad(x.shape[2], kh, 1)
  pl, pr = O.same_pad(x.shape[3], kw, 1)
  xp = F.pad(x, (pl, pr, pt, pb))
  w = k.permute(3, 2, 0, 1).contiguous()
  return torch.cat([F.conv2d(xp[:, :, r0:r0 + rows + kh - 1], w, b) for r0 in range(0, x.shape[2], rows)], 2)


def _softmax_bound(lg, kernel):
  """float64 softmax of the device's float32 logits [N, NC] and the largest |p_dev - p| the kernel may show.

  With a_c the base-2 exponent argument and da_c its error (SOFTMAX_ERR), the kernel's unnormalised terms are
  e'_c = 2^(a_c + da_c) (1 +- e_exp); the fp32 sum of NC positive terms adds (NC - 1) u, the reciprocal and the final
  product e_div.  So |p'_c / p_c - 1| <= (1 + r_c)(1 + e_div) / (1 - sum_j p_j r_j - (NC - 1) u) - 1 with
  r_c = 2^|da_c| (1 + e_exp) - 1.  ex2.approx.ftz flushes results below 2^-126: 2^-120 absolute covers that."""
  ka, km, e_exp, e_div = SOFTMAX_ERR[kernel]
  l = lg.astype(np.float64)
  mx = l.max(-1, keepdims=True)
  e = np.exp(l - mx)
  p = e / e.sum(-1, keepdims=True)
  da = u * LOG2E * (ka * np.abs(l - mx) + km * np.abs(mx))
  r = np.exp2(da) * (1.0 + e_exp) - 1.0
  rs = (p * r).sum(-1, keepdims=True) + (l.shape[-1] - 1) * u
  rel = (1.0 + r) * (1.0 + e_div) / (1.0 - rs) - 1.0
  return p, rel * p * (1.0 + 1e-6) + 2.0 ** -120


def _guarded(n, dtype, fill, sentinel):
  t = torch.full((n + 2 * GUARD,), sentinel, dtype=dtype, device="cuda")
  t[GUARD:GUARD + n] = fill
  return t


def _ptr(t):
  return None if t is None else t.data_ptr() + GUARD * t.element_size()


def _split(t, n):
  """(interior, guards) of a guarded buffer as numpy; guards as raw bits."""
  a = t.cpu().numpy()
  bits = a.view(np.int32)
  return a[GUARD:GUARD + n], np.concatenate([bits[:GUARD], bits[GUARD + n:]])


class Case:
  def __init__(self, c, seed):
    self.c = c
    self.nc, self.H, self.W, self.B = c["nc"], c["H"], c["W"], c["B"]
    self.none_index = 0 if c["none"] == "0" else self.nc - 1
    self.n_px = self.B * self.H * self.W
    rng = np.random.default_rng(seed)
    g = self.g = L.Graph(self.H, self.W)
    g.rng = np.random.default_rng(seed + 1)
    self.a = L.relu(L.BatchNormalization("b0")(L.Conv2D("c0", c["cin"], 3)(g.input)))
    h = L.BatchNormalization("bh")(L.Conv2D("head", self.nc, c["k"])(self.a))
    if c["act"] == "relu":
      h = L.relu(h)
    elif c["act"] == "leaky":
      h = L.LeakyReLU(0.1)(h)
    self.head = h
    _rand_vars(g, rng)
    _head_weights(g, c["weights"])
    x = rng.normal(size=(self.B, self.H, self.W, 6)).astype(np.float32)
    x[..., 5] = rng.random((self.B, self.H, self.W)) < 0.8
    self.x = _f16(x)
    self.mask = (rng.random((self.B, self.H, self.W)) < 0.7).astype(np.uint8)
    differ = (self.mask != (self.x[..., 5] != 0)).mean()
    assert differ > 0.2, differ                        # the kernels must follow the mask array, not channel 5
    self.x_d = torch.from_numpy(self.x).cuda()
    self.mask_d = torch.from_numpy(self.mask).cuda()
    self.lib = _lib.load()

  def build(self, **opts):
    o = {"conv_impl": self.c["impl"], "use_graph": 0, "keep_tensors": 1}
    if self.c["mb"]:
      o["micro_batch"] = self.c["mb"]
    o.update(opts)
    return self.g.build_net(self.head, self.nc, self.none_index, PREC[self.c["prec"]], self.B, o)

  def buffers(self, want=True):
    n = self.n_px * self.nc
    lg = _guarded(n, torch.float32, float("nan"), float(F_SENT)) if want else None
    pr = _guarded(n, torch.float32, float("nan"), float(F_SENT)) if want else None
    pd = _guarded(self.n_px, torch.int32, -7, I_SENT)
    return lg, pr, pd

  def forward(self, net, bufs):
    lg, pr, pd = bufs
    _lib.check(self.lib.pcls_net_forward(net, self.x_d.data_ptr(), 6, self.mask_d.data_ptr(), None, None, self.B,
                                         _ptr(lg), _ptr(pr), _ptr(pd), torch.cuda.current_stream().cuda_stream),
               "pcls_net_forward")
    torch.cuda.synchronize()

  def outputs(self, bufs):
    """(logits, probs, preds) as [B,H,W,(NC)] numpy after checking the guard bands and that every element was written."""
    lg, pr, pd = bufs
    out = []
    for t, n, what in ((lg, self.n_px * self.nc, "logits"), (pr, self.n_px * self.nc, "probs"), (pd, self.n_px, "preds")):
      if t is None:
        out.append(None)
        continue
      inner, guards = _split(t, n)
      sent = I_SENT if what == "preds" else int(np.array([F_SENT]).view(np.int32)[0])
      assert (guards == sent).all(), "%s: %d guard elements overwritten" % (what, int((guards != sent).sum()))
      if what == "preds":
        assert (inner != -7).all(), "preds: %d pixels never written" % int((inner == -7).sum())
        out.append(inner.reshape(self.B, self.H, self.W))
      else:
        assert not np.isnan(inner).any(), "%s: %d elements never written (or NaN)" % (what, int(np.isnan(inner).sum()))
        out.append(inner.reshape(self.B, self.H, self.W, self.nc))
    return out


def _kernel_sequence(case, net, bufs):
  """Runs the forward once under torch.profiler; returns the names of the project's kernels in launch order."""
  from torch.profiler import ProfilerActivity, profile
  torch.cuda.synchronize()
  with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
    case.forward(net, bufs)
  evs = sorted((e for e in prof.events() if KERNEL_RE.search(e.name)),
               key=lambda e: e.time_range.start)
  return [e.name for e in evs]


def _head_inst(name):
  """(KC, CS, is_bf16) of a conv_head_kernel name, demangled or mangled."""
  m = re.search(r"conv_head_kernel<\s*([\w:]+)\s*,\s*(\d+)\s*,\s*(\d+)\s*>", name) or \
      re.search(r"conv_head_kernelI(\w+?)Li(\d+)ELi(\d+)E", name)
  assert m, "cannot read the template arguments of %r" % name
  return int(m.group(2)), int(m.group(3)), "bfloat16" in m.group(1)


def _check_path(case, names, lpf):
  c = case.c
  passes = -(-case.B // c["mb"]) if c["mb"] else 1
  unfused = c["path"] in ("C", "D")
  assert lpf == (4 if unfused else 3), "launches per forward %d: path %s expects %s head" % (
      lpf, c["path"], "a standalone" if unfused else "a fused")
  assert len(names) == passes * lpf, "%d passes x %d launches expected, profiled %s" % (passes, lpf, names)
  for i in range(passes):
    seq = names[i * lpf:(i + 1) * lpf]
    assert "net_input_kernel" in seq[0], seq
    logits_k = seq[2]
    for path, kern in PATH_KERNEL.items():   # the logits layer ran the kernel of the claimed path, and only that one
      if kern != PATH_KERNEL[c["path"]]:
        assert kern not in logits_k, "logits layer ran %r: this case claims path %s" % (logits_k, c["path"])
    assert PATH_KERNEL[c["path"]] in logits_k, "logits layer ran %r: this case claims path %s" % (logits_k, c["path"])
    if c["path"] == "A":
      kc, cs, bf = _head_inst(logits_k)
      assert (kc, cs) == c["inst"] and bf == (c["prec"] == "bf16"), (logits_k, c["inst"], c["prec"])
    if unfused:   # (conv_head_kernel contains the substring head_kernel)
      assert "head_kernel" in seq[3] and "conv_head_kernel" not in seq[3], seq
    else:
      assert not any(re.search(r"(?<!conv_)head_kernel", n) for n in seq), seq


def _check_regime(case):
  c = case.c
  sms = torch.cuda.get_device_properties(0).multi_processor_count
  n_wt = -(-case.W // HD_TILE)
  frames = c["mb"] or case.B
  tiles = n_wt * case.H * frames
  grid = min(tiles, sms)
  per_cta, stride, frame = tiles / grid, HD_NG * grid, n_wt * case.H
  what = "%d tiles, %d SMs, %.1f tiles per CTA, group stride %d tiles, frame %d tiles" % (tiles, sms, per_cta, stride, frame)
  if c["regime"] == "few":
    assert tiles < sms, what
  elif c["regime"] == "1-4":
    assert 1 < per_cta <= 4, what
  elif c["regime"] == "wrap-in-frame":
    assert per_cta > 2 * 8 and stride < frame, what
  elif c["regime"] == "wrap-frames":
    assert per_cta > 2 * 8 and stride >= 2 * frame, what


def _check_probs(what, lg, pr, kernel, nc):
  """Check 2 on every pixel: pr against the float64 softmax of lg."""
  l2, p2 = lg.reshape(-1, nc), pr.reshape(-1, nc)
  assert np.isfinite(l2).all(), "%s: non-finite logits" % what
  assert np.isfinite(p2).all() and (p2 >= 0).all(), "%s: probabilities not finite / negative" % what
  p64, bound = _softmax_bound(l2, kernel)
  d = np.abs(p2.astype(np.float64) - p64)
  worst = float((d / bound).max())
  assert worst <= 1.0, "%s: probability error %.3g x the %s softmax bound (max abs err %.3e)" % (what, worst, kernel, d.max())
  # every row sums to 1 within the bound: the padding classes (there are CS - NC or 32 - NC of them) carry no mass
  srow = np.abs(p2.astype(np.float64).sum(-1) - 1.0)
  assert (srow <= bound.sum(-1) + nc * 2.0 ** -52).all(), "%s: a probability row sums to 1 %+.3e" % (what, srow.max())


def _check_preds(what, case, pr, pd):
  """Check 3 on every pixel."""
  m = case.mask.astype(bool)
  assert ((pd >= 0) & (pd < case.nc)).all(), "%s: predictions outside [0, NC)" % what
  assert (pd[~m] == case.none_index).all(), "%s: masked pixels not none_index" % what
  am = np.argmax(pr, -1)   # numpy: first index on ties, like the kernels
  bad = (pd != am) & m
  assert not bad.any(), "%s: %d predictions differ from argmax(probs), first at %s: pred %d, probs %s" % (
      what, int(bad.sum()), np.argwhere(bad)[0], pd[tuple(np.argwhere(bad)[0])], pr[tuple(np.argwhere(bad)[0])])


@pytest.mark.parametrize("c", CASES)
def test_logits_and_head_against_float64(c, request):
  case = Case(c, seed=zlib.crc32(request.node.callspec.id.encode()))
  lib = case.lib
  U = U16[c["prec"]]
  if c["path"] == "A":
    _check_regime(case)
  net = case.build()
  try:
    # ---- one forward under the profiler: the kernels, then the outputs of that same forward ----
    bufs = case.buffers()
    names = _kernel_sequence(case, net, bufs)
    _check_path(case, names, lib.pcls_net_launches_per_forward(net))
    lg, pr, pd = case.outputs(bufs)                                           # check 4
    soft = {"A": "conv_head", "B": "conv_tc"}.get(c["path"], "head")
    _check_probs("fused" if soft != "head" else "head_kernel", lg, pr, soft, case.nc)  # check 2
    _check_preds("forward", case, pr, pd)                                       # check 3

    # ---- check 1: logits vs float64 on the device's own c0 output (the last pass's frames when micro-batched) ----
    nb = (case.B - (case.B - 1) // c["mb"] * c["mb"]) if c["mb"] else case.B
    frames = [nb - 1] if c["mb"] else sorted({0, case.B - 1})
    gframes = [case.B - nb + f for f in frames]
    xa = torch.empty((nb, case.H, case.W, c["cin"]), dtype=torch.float32, device="cuda")
    _lib.check(lib.pcls_net_read_tensor(net, case.a.tid, nb, xa.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "read c0")
    torch.cuda.synchronize()
    x = torch.from_numpy(xa.cpu().numpy()[frames]).permute(0, 3, 1, 2).double()
    p = {k: torch.from_numpy(v) for k, v in case.g.variables.items()}
    k, b = _fold64(p, "head", "bh")
    y = _conv_same_rows(x, k, b)
    S = _conv_same_rows(x.abs(), k.abs(), b.abs())
    if c["act"] == "relu":
      y = torch.relu(y)
    elif c["act"] == "leaky":
      y = O.leaky(y)
    y = y.permute(0, 2, 3, 1).numpy()
    bound = U * 1.5 * S.permute(0, 2, 3, 1).numpy() + 2.0 ** -22 * np.abs(y) + 1e-6
    d = np.abs(lg[gframes].astype(np.float64) - y)
    worst = float((d / bound).max())
    assert worst <= 1.0, "logits: error %.3g x the error model (max abs err %.3e)" % (worst, d.max())
    if c["weights"] == "large":
      assert np.abs(lg).max() > 300.0, np.abs(lg).max()
    # labels: wherever the oracle's two best logits are further apart than twice the logit bound
    top2 = np.sort(y, -1)[..., -2:]
    m = case.mask[gframes].astype(bool)
    decidable = m & (top2[..., 1] - top2[..., 0] > 2 * bound.max(-1))
    wrong = decidable & (pd[gframes] != np.argmax(y, -1))
    assert not wrong.any(), "%d decidable pixels disagree with the oracle's label" % int(wrong.sum())
    if c["weights"] == "rand":
      assert decidable.sum() > 0.5 * m.sum(), (int(decidable.sum()), int(m.sum()))

    # ---- semantics the case was built for ----
    mm = case.mask.astype(bool)
    if c["weights"] == "zero":                  # every class has the same logit: class 0 on every unmasked pixel
      assert (pd[mm] == 0).all() and (pr == pr[..., :1]).all()
    if c["weights"] == "ties":                  # the duplicated classes tie exactly; the lower index must win
      for i, j in TIE_PAIRS:
        assert np.array_equal(lg[..., i], lg[..., j]) and np.array_equal(pr[..., i], pr[..., j])
        won = mm & (np.argmax(np.delete(pr, j, -1), -1) == i)
        assert won.sum() > 0.03 * mm.sum(), int(won.sum())
        assert (pd[won] == i).all()

    # ---- check 5: other plumbing ----
    b2 = case.buffers(want=False)                                              # the benchmark's call: preds only
    case.forward(net, b2)
    assert np.array_equal(case.outputs(b2)[2], pd), "logits = probs = NULL changes the predictions"

    net2 = case.build(keep_tensors=0, micro_batch=0) if c["mb"] else case.build(keep_tensors=0)
    try:
      b3 = case.buffers()
      case.forward(net2, b3)
      lg3, pr3, pd3 = case.outputs(b3)
      what = "micro_batch = 0, keep_tensors = 0" if c["mb"] else "keep_tensors = 0"
      assert np.array_equal(lg3, lg) and np.array_equal(pr3, pr) and np.array_equal(pd3, pd), what + ": outputs differ"
    finally:
      lib.pcls_net_destroy(net2)

    _lib.check(lib.pcls_net_set_option(net, b"fuse_head", 0), "fuse_head = 0")
    assert lib.pcls_net_launches_per_forward(net) == 4           # logits layer + standalone head_kernel
    b4 = case.buffers()
    case.forward(net, b4)
    lg4, pr4, pd4 = case.outputs(b4)
    assert np.array_equal(lg4.view(np.int32), lg.view(np.int32)), "fuse_head = 0: logits not bit-identical"
    _check_probs("fuse_head = 0 (head_kernel)", lg4, pr4, "head", case.nc)
    _check_preds("fuse_head = 0", case, pr4, pd4)
    if soft == "head":
      assert np.array_equal(pr4, pr) and np.array_equal(pd4, pd)            # the same kernels ran
    else:
      # a label may differ only where the two best logits are closer than the two softmax bounds together
      flip = pd4 != pd
      if flip.any():
        lf, a, b = lg[flip], pd[flip][:, None], pd4[flip][:, None]
        p64, bf = _softmax_bound(lf, soft)
        _, bh = _softmax_bound(lf, "head")
        rel = (bf + bh) / p64      # relative error of either probability, per class
        tol = np.take_along_axis(rel, a, -1) + np.take_along_axis(rel, b, -1)
        gap = np.abs(np.take_along_axis(lf, a, -1) - np.take_along_axis(lf, b, -1))
        assert (gap <= tol).all(), "fuse_head = 0 flips %d labels beyond float rounding" % int(flip.sum())
  finally:
    lib.pcls_net_destroy(net)
