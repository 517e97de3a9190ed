"""numpy restatement of the MC-dropout rules of include/pclseg.h (TEST INFRASTRUCTURE ONLY - never imported by the
product): the Philox4x32-10 generator, the dropout mask and its bit-exact application to fp16 / bf16 tensors, a float64
dropout for the network oracle, the accumulate / finalize rules over T passes, and the binned AUROC of
``metrics.UncertaintyAUROC``.  ``forward`` is ``oracle.nn.forward`` with the dropout sites of the two architectures
applied in place (SqueezeSegV2: site 0 = fire13 + conv1_skip; Darknet: sites 0-4 = enc1 .. enc5, site 5 = the head's
input), built from ``oracle.nn``'s own layer functions."""
from __future__ import annotations

import numpy as np
import torch

from . import nn as onn

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
  """ctr [..., 4], key [..., 2] (anything that converts to uint64, values < 2^32) -> [..., 4] uint64 output words."""
  c = [np.asarray(ctr, np.uint64)[..., i] for i in range(4)]
  k = [np.asarray(key, np.uint64)[..., i] for i in range(2)]
  k = [np.broadcast_to(k[0], c[0].shape).copy(), np.broadcast_to(k[1], c[0].shape).copy()]
  for r in range(10):
    if r:
      k = [(k[0] + W0) & MASK32, (k[1] + W1) & MASK32]
    p0, p1 = M0 * c[0], M1 * c[2]                      # < 2^64: exact in uint64
    hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
    hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
    c = [hi1 ^ c[1] ^ k[0], lo1, hi0 ^ c[3] ^ k[1], lo0]
  return np.stack(c, axis=-1)


def threshold(rate):
  thr = int(np.floor(float(rate) * 65536.0 + 0.5))
  if not (rate >= 0 and thr < 65536):
    raise ValueError("invalid rate %r" % rate)
  return thr


def scale_of(thr):
  return np.float32(65536.0 / (65536 - thr))


def uniforms(seed, frame, n_pass, site, n_elements):
  """The 16-bit u of elements 0 .. n_elements-1 (a multiple of 8) of one frame's tensor, uint32 [n_elements]."""
  g = np.arange(n_elements // 8, dtype=np.uint64)
  ctr = np.stack([g, np.full_like(g, site | (n_pass << 16)), np.full_like(g, frame & 0xFFFFFFFF),
                  np.full_like(g, frame >> 32)], axis=-1)
  w = philox4x32_10(ctr, [seed & 0xFFFFFFFF, seed >> 32])            # [G, 4]
  u = np.stack([w & np.uint64(0xFFFF), w >> np.uint64(16)], axis=-1)  # [G, 4, 2]: element 8g + 2i + j
  return u.reshape(-1).astype(np.uint32)


def keep_mask(seed, frame_base, n_pass, site, rate, shape):
  """bool keep mask of a [B, H, W, C] tensor whose frame b has the global id frame_base + b."""
  B = shape[0]
  n = int(np.prod(shape[1:]))
  thr = threshold(rate)
  return np.stack([uniforms(seed, frame_base + b, n_pass, site, n) >= thr for b in range(B)]).reshape(shape)


def to_f32(bits, dtype):
  bits = np.asarray(bits, np.uint16)
  if dtype == "f16":
    return bits.view(np.float16).astype(np.float32)
  return (bits.astype(np.uint32) << np.uint32(16)).view(np.float32)


def from_f32(x, dtype):
  x = np.asarray(x, np.float32)
  if dtype == "f16":
    return x.astype(np.float16).view(np.uint16)
  b = x.view(np.uint32).astype(np.uint64)
  return ((b + np.uint64(0x7FFF) + ((b >> np.uint64(16)) & np.uint64(1))) >> np.uint64(16)).astype(np.uint16)


def dropout_bits(bits, dtype, seed, frame_base, n_pass, site, rate):
  """The dropout of a 16-bit tensor [B, H, W, C] (uint16 bit patterns, dtype "f16" | "bf16"), bit-exact: kept
  elements become round16(fl32(x) * scale), dropped ones the bit pattern 0."""
  bits = np.asarray(bits, np.uint16)
  keep = keep_mask(seed, frame_base, n_pass, site, rate, bits.shape)
  with np.errstate(invalid="ignore", over="ignore"):
    y = from_f32(to_f32(bits, dtype) * scale_of(threshold(rate)), dtype)
  return np.where(keep, y, np.uint16(0))


def apply_dropout(x_nhwc, seed, frame_base, n_pass, site, rate):
  """float64 dropout for the network oracle: x * keep * scale (scale as the kernel's float32 value)."""
  keep = keep_mask(seed, frame_base, n_pass, site, rate, x_nhwc.shape)
  return np.where(keep, np.asarray(x_nhwc, np.float64) * float(scale_of(threshold(rate))), 0.0)


def entropy(p, nc):
  """Normalised entropy by the kernels' rule (float32, class order, over p > 0, divided by logf(NC)); numpy's float32
  log may differ from the device's logf in the last bit, so compare with a bound."""
  p = np.asarray(p, np.float32)
  h = np.zeros(p.shape[:-1], np.float32)
  for c in range(nc):
    pc = p[..., c]
    term = np.where(pc > 0, pc * np.log(np.where(pc > 0, pc, 1)).astype(np.float32), 0).astype(np.float32)
    h = (h + term).astype(np.float32)
  return (-h / np.float32(np.log(np.float32(nc)))).astype(np.float32) if nc > 1 else np.zeros_like(h)


def accumulate(probs_list):
  """(acc_probs float32, acc_entropy float64) over the passes' probabilities [..., NC], in pass order."""
  nc = probs_list[0].shape[-1]
  acc_p = np.asarray(probs_list[0], np.float32).copy()
  acc_h = entropy(probs_list[0], nc).astype(np.float64)
  for p in probs_list[1:]:
    acc_p = (acc_p + np.asarray(p, np.float32)).astype(np.float32)
    acc_h = acc_h + entropy(p, nc).astype(np.float64)
  return acc_p, acc_h


def finalize(acc_p, acc_h, mask, n_passes, none_index):
  """dict(probabilities, predictions, confidence, entropy, mutual_information) by the pcls_mc_finalize rules."""
  nc = acc_p.shape[-1]
  mean = (np.asarray(acc_p, np.float32) / np.float32(n_passes)).astype(np.float32)
  pred = np.argmax(mean, axis=-1).astype(np.int32)          # first index on ties
  valid = np.ones(pred.shape, bool) if mask is None else np.asarray(mask) != 0
  H = entropy(mean, nc)
  EH = (np.asarray(acc_h, np.float64) / n_passes).astype(np.float32)
  mi = np.maximum(np.float32(0), (H - EH).astype(np.float32))
  return dict(probabilities=mean, predictions=np.where(valid, pred, none_index).astype(np.int32),
              confidence=np.where(valid, mean.max(axis=-1), 0).astype(np.float32),
              entropy=np.where(valid, H, 0).astype(np.float32),
              mutual_information=np.where(valid, mi, 0).astype(np.float32))


def binned_auroc(count, correct):
  """AUROC of an uncertainty u for detecting errors from a histogram of u: per bin the number of elements and of correct
  ones.  An (error, correct) pair counts 1 when the error's bin is above the correct one's, 1/2 in the same bin.
  0.5 when either class is empty."""
  count = np.asarray(count, np.float64)
  correct = np.asarray(correct, np.float64)
  err = count - correct
  n_err, n_ok = err.sum(), correct.sum()
  if n_err == 0 or n_ok == 0:
    return 0.5
  below_ok = np.concatenate([[0.0], np.cumsum(correct)[:-1]])
  return float((err * (below_ok + 0.5 * correct)).sum() / (n_err * n_ok))


def forward(arch, params, lidar_bhw6, mask_bhw, none_index, dropout, num_layers=53, output_stride=16,
            dtype=torch.float64):
  """``oracle.nn.forward`` with ``dropout(site, x_nhwc numpy) -> numpy`` applied at every site, in place."""
  p = {k: (v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v))).to(dtype) for k, v in params.items()}
  x = torch.as_tensor(np.asarray(lidar_bhw6)).to(dtype).permute(0, 3, 1, 2).contiguous()

  def drop(site, t):
    y = dropout(site, t.permute(0, 2, 3, 1).cpu().numpy())
    return torch.as_tensor(np.asarray(y)).to(dtype).permute(0, 3, 1, 2).contiguous()

  F_relu = torch.nn.functional.relu
  if arch == "squeezesegv2":
    y = F_relu(onn.batch_norm(onn._conv(x, p, "conv1", (1, 2)), p, "bn1"))
    cam1 = onn.cam(y, p, "cam1")
    skip = onn.batch_norm(onn._conv(x, p, "conv1_skip"), p, "bn1_skip")
    y = onn.fire(onn.max_pool_same(cam1, 3, (1, 2)), p, "fire2")
    y = onn.fire(onn.cam(y, p, "cam2"), p, "fire3")
    cam3 = onn.cam(y, p, "cam3")
    fire5 = onn.fire(onn.fire(onn.max_pool_same(cam3, 3, (1, 2)), p, "fire4"), p, "fire5")
    y = onn.max_pool_same(fire5, 3, (1, 2))
    for name in ("fire6", "fire7", "fire8", "fire9"):
      y = onn.fire(y, p, name)
    y = onn.fireup(y, p, "fire10") + fire5
    y = onn.fireup(y, p, "fire11") + cam3
    y = onn.fireup(y, p, "fire12") + cam1
    y = drop(0, onn.fireup(y, p, "fire13") + skip)
    logits = onn._conv(y, p, "conv14")
  elif arch == "darknet":
    enc_s, dec_s = onn.darknet_strides(output_stride)
    nb = onn.MODEL_BLOCKS[num_layers]
    skips, os_ = {}, 1
    y = onn.leaky(onn.batch_norm(onn._conv(x, p, "conv1"), p, "bn1"))
    for i in range(5):
      z = onn.encoder_layer(y, p, f"enc{i + 1}", nb[i], enc_s[i])
      if z.shape[2] < y.shape[2] or z.shape[3] < y.shape[3]:
        skips[os_] = y
        os_ *= 2
      y = drop(i, z)
    for j, i in enumerate([5, 4, 3, 2, 1]):
      z = onn.decoder_layer(y, p, f"dec{i}", dec_s[j])
      if z.shape[3] > y.shape[3]:
        os_ //= 2
        z = z + skips[os_]
      y = z
    logits = onn._conv(drop(5, y), p, "head")
  else:
    raise ValueError(arch)
  logits = logits.permute(0, 2, 3, 1).contiguous()
  prob, pred = onn.segmentation_head(logits, torch.as_tensor(np.asarray(mask_bhw)), none_index)
  return logits.numpy(), prob.numpy(), pred.numpy()
