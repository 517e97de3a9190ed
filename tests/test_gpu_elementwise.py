"""Head, input stage and confusion matrix through the C ABI vs the oracle."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import confusion as C
from oracle import nn as O
from pclsegmentation_b200 import _lib
from tests.util import synth_range_images

pytestmark = pytest.mark.gpu


def _s():
  return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("n,nc,none", [(64 * 2048 * 2, 20, 0), (32 * 240 * 3 + 7, 11, 10), (5, 3, 1), (33, 32, 31)])
def test_head_matches_oracle(n, nc, none):
  lib = _lib.load()
  rng = np.random.default_rng(n)
  logits = (rng.normal(size=(n, nc)) * 4).astype(np.float32)
  logits[::7] = np.round(logits[::7])            # exact ties -> lowest index must win
  logits[1::11, :] = 3.0
  mask = rng.random(n) < 0.7
  lg, m = torch.from_numpy(logits).cuda(), torch.from_numpy(mask).cuda()
  probs = torch.empty_like(lg)
  preds = torch.empty(n, dtype=torch.int32, device="cuda")
  _lib.check(lib.pcls_head(lg.data_ptr(), m.view(torch.uint8).data_ptr(), n, nc, none, probs.data_ptr(),
                           preds.data_ptr(), _s()))
  p_ref, pred_ref = O.segmentation_head(torch.from_numpy(logits), torch.from_numpy(mask), none)
  assert np.allclose(probs.cpu().numpy(), p_ref.numpy(), rtol=2e-6, atol=1e-7)
  got = preds.cpu().numpy()
  # argmax is taken over OUR rounded probabilities: it must equal the reference wherever the oracle's top-2
  # probabilities are not within float rounding of each other, and always be a maximiser of our own probabilities
  top2 = np.sort(p_ref.numpy(), axis=1)[:, -2:]
  clear = (top2[:, 1] - top2[:, 0]) > 1e-6
  assert np.array_equal(got[clear | ~mask], pred_ref.numpy()[clear | ~mask])
  own = probs.cpu().numpy()
  assert np.array_equal(got[mask], own.argmax(1)[mask])
  assert (got == pred_ref.numpy()).mean() > 0.9999
  # probs = NULL variant gives the same predictions
  preds2 = torch.empty_like(preds)
  _lib.check(lib.pcls_head(lg.data_ptr(), m.view(torch.uint8).data_ptr(), n, nc, none, None, preds2.data_ptr(), _s()))
  assert torch.equal(preds, preds2)


def test_input_stage_matches_oracle():
  from pclsegmentation_b200.configs import SqueezeSegV2KittiConfig
  lib = _lib.load()
  mc = SqueezeSegV2KittiConfig()
  rng = np.random.default_rng(1)
  raw = synth_range_images(rng, 2, 64, 512)
  n = 2 * 64 * 512
  d = torch.from_numpy(raw).cuda()
  lidar = torch.empty((n, 6), dtype=torch.float32, device="cuda")
  mask = torch.empty(n, dtype=torch.uint8, device="cuda")
  label = torch.empty(n, dtype=torch.int32, device="cuda")
  mean = (ctypes.c_double * 5)(*mc.INPUT_MEAN.reshape(-1))
  std = (ctypes.c_double * 5)(*mc.INPUT_STD.reshape(-1))
  weight = torch.empty(n, dtype=torch.float32, device="cuda")
  cls_w = np.linspace(0.25, 3.0, mc.NUM_CLASS)          # distinct per class (the shipped configs use ones / a 0 for None)
  cw = (ctypes.c_double * mc.NUM_CLASS)(*cls_w)
  raw[0, :4, :8, 5] = 25.0                              # labels outside [0, NUM_CLASS): weight stays 0 (np.zeros)
  raw[0, :4, :8, 4] = 5.0
  d = torch.from_numpy(raw).cuda()
  _lib.check(lib.pcls_input_stage(d.data_ptr(), 6, n, mean, std, 0, lidar.data_ptr(), mask.data_ptr(),
                                  label.data_ptr(), cw, mc.NUM_CLASS, weight.data_ptr(), _s()))
  for b in range(2):
    l_ref, m_ref, lab_ref = O.input_stage(raw[b], mc.INPUT_MEAN, mc.INPUT_STD, 0)
    sl = slice(b * 64 * 512, (b + 1) * 64 * 512)
    assert np.array_equal(lidar[sl].cpu().numpy().reshape(64, 512, 6), l_ref)     # bit-exact (float64 normalise)
    assert np.array_equal(mask[sl].cpu().numpy().reshape(64, 512).astype(bool), m_ref)
    assert np.array_equal(label[sl].cpu().numpy().reshape(64, 512), lab_ref)
    w_ref = O.class_weight_map(O.fixed_label(raw[b], 0), cls_w)                   # data_loader.py:181-185 (float label)
    assert np.array_equal(weight[sl].cpu().numpy().reshape(64, 512), w_ref)
  assert (weight.cpu().numpy().reshape(2, 64, 512)[0, :4, :8] == 0).all()
  # the DataLoader.parse_sample facade returns the same four arrays
  from pclsegmentation_b200.data_loader import parse_samples
  mc.CLS_LOSS_WEIGHT = cls_w
  lid, msk, lab, wgt = parse_samples(raw, mc)
  assert np.array_equal(lid.cpu().numpy(), lidar.cpu().numpy().reshape(2, 64, 512, 6)) and msk.dtype == torch.bool
  assert np.array_equal(lab.cpu().numpy().ravel(), label.cpu().numpy()) and np.array_equal(wgt.cpu().numpy().ravel(), weight.cpu().numpy())


@pytest.mark.parametrize("n,nc", [(32 * 64 * 2048, 20), (3 * 32 * 240 + 3, 11), (1, 2), (0, 11)])
def test_confusion_bit_exact(n, nc):
  from pclsegmentation_b200.metrics import MeanIoU
  from pclsegmentation_b200.utils.util import confusion_matrix_to_iou_recall_precision
  rng = np.random.default_rng(n + nc)
  p = np.full(nc, 0.5 / max(nc - 1, 1))
  p[nc - 1] = 0.5                                 # heavily skewed, like the None class
  p /= p.sum()
  label = rng.choice(nc, n, p=p).astype(np.int32)
  pred = np.where(rng.random(n) < 0.8, label, rng.integers(0, nc, n)).astype(np.int32)
  m = MeanIoU(nc)
  half = (n // 2) // 4 * 4
  m.update_state(label[:half], pred[:half])       # accumulates across calls like update_state
  m.update_state(label[half:], pred[half:])
  ref = C.confusion_matrix(label, pred, nc)
  assert np.array_equal(m.total_cm.cpu().numpy(), ref) and m.dropped == 0
  assert abs(float(m.result()) - C.mean_iou(ref)) < 1e-6
  got = confusion_matrix_to_iou_recall_precision(m.total_cm)
  assert all(np.allclose(a, b) for a, b in zip(got, C.iou_recall_precision(ref)))
  m.reset_states()
  assert int(m.total_cm.sum()) == 0


def test_confusion_out_of_range_pairs_are_dropped_and_counted():
  from pclsegmentation_b200.metrics import MeanIoU
  m = MeanIoU(4)
  m.update_state(np.array([0, 1, 7, -1, 2], np.int32), np.array([0, 9, 1, 1, 2], np.int32))
  assert int(m.total_cm.sum()) == 2 and m.dropped == 3


@pytest.mark.gpu
def test_test_step_losses_and_weighted_miou():
  """test_step (nets/SegmentationNetwork.py:118-131): focal loss (:71-91), Keras sparse categorical cross-entropy on
  probabilities with sample weights (:49), running mean of the loss, weighted confusion matrix - against float64 numpy
  restatements of the same formulas on the probabilities / predictions the GPU forward returned."""
  from pclsegmentation_b200.utils.args_loader import load_model_config
  from tests.util import synth_range_images
  from oracle import nn as O
  mc, model = load_model_config("squeezesegv2", "squeezesegv2")
  model.randomize_batch_norm(2)
  H, W, NC = mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL, mc.NUM_CLASS
  rng = np.random.default_rng(5)
  raw = synth_range_images(rng, 2, H, W, valid_rate=0.7, num_classes=NC)
  lidar, mask, label = [], [], []
  for b in range(raw.shape[0]):
    l, m, y = O.input_stage(raw[b], mc.INPUT_MEAN, mc.INPUT_STD, mc.CLASSES.index("None"))
    lidar.append(l); mask.append(m); label.append(y)
  lidar, mask, label = np.stack(lidar), np.stack(mask), np.stack(label).astype(np.int32)
  weight = np.asarray(mc.CLS_LOSS_WEIGHT, np.float32)[label] if hasattr(mc, "CLS_LOSS_WEIGHT") else \
      rng.uniform(0.5, 2.0, label.shape).astype(np.float32)
  probs, preds = model([lidar, mask])
  p = probs.numpy().astype(np.float64).reshape(-1, NC)
  y = label.reshape(-1)
  w = weight.astype(np.float64).reshape(-1)
  m = mask.astype(np.float64).reshape(-1)
  # focal loss
  pe = p + mc.DENOM_EPSILON
  onehot = np.eye(NC)[y]
  fl = ((1.0 - pe) ** mc.FOCAL_GAMMA * onehot * -np.log(pe) * w[:, None] * m[:, None]).sum() / m.sum() * mc.CLS_LOSS_COEF
  got_fl = float(model.focal_loss(probs, mask, label, weight))
  assert abs(got_fl - fl) <= 2e-5 * max(1.0, abs(fl)), (got_fl, fl)
  # sparse categorical cross-entropy (Keras: clip, renormalise, weight, mean over all elements)
  pc = np.clip(p, 1e-7, 1 - 1e-7)
  scc = (-(np.log(pc[np.arange(len(y)), y]) - np.log(pc.sum(1))) * w).sum() / len(y)
  got_scc = float(model.scc_loss(label, probs, weight))
  assert abs(got_scc - scc) <= 2e-5 * max(1.0, abs(scc)), (got_scc, scc)
  # test_step: running mean of the loss over two steps + weighted MeanIoU
  model.miou_tracker.reset_states()
  r1 = model.test_step(((lidar, mask), label, weight))
  r2 = model.test_step(((lidar, mask), label, weight))
  expect = fl if mc.USE_FOCAL_LOSS else scc
  assert abs(float(r1["loss"]) - expect) <= 1e-4 * max(1.0, abs(expect))
  assert abs(float(r2["loss"]) - expect) <= 1e-4 * max(1.0, abs(expect))
  cm = np.zeros((NC, NC))
  np.add.at(cm, (y, preds.numpy().reshape(-1)), w)
  got_cm = model.miou_tracker.total_cm.cpu().numpy()
  assert np.allclose(got_cm, 2 * cm, rtol=1e-9, atol=1e-6)
  tp = np.diag(cm); den = cm.sum(0) + cm.sum(1) - tp
  assert abs(float(r2["miou"]) - (tp[den > 0] / den[den > 0]).mean()) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 7, 4096, 32 * 240 * 6 * 3 + 1])
def test_cast_f64_f32_is_numpy_astype(n):
  """pcls_cast_f64_f32 == numpy's astype(float32) bit for bit (round to nearest even), incl. values that are not
  representable in float32, subnormals, infinities and odd lengths."""
  rng = np.random.default_rng(n)
  x = rng.normal(0, 50, n)
  if n >= 7:
    x[:7] = [0.1, -1e-45, 3.4028235677973366e38, 1e39, -np.inf, 16777217.0, 1.0000000596046448]
  d = torch.from_numpy(x).cuda()
  out = torch.empty(n, dtype=torch.float32, device="cuda")
  lib = _lib.load()
  with np.errstate(over="ignore"):
    want = x.astype(np.float32)
  _lib.check(lib.pcls_cast_f64_f32(d.data_ptr(), out.data_ptr(), n, torch.cuda.current_stream().cuda_stream))
  got = out.cpu().numpy()
  assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
  from pclsegmentation_b200.device import samples_to_device
  if n > 0:
    t = samples_to_device(x.reshape(1, 1, 1, n))
    assert t.dtype == torch.float32 and np.array_equal(t.cpu().numpy().reshape(-1).view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("n,nc", [(32 * 240 * 2 + 5, 11), (64 * 2048 + 1, 20), (31, 3), (1, 32), (0, 11)])
def test_validation_kernel_against_float64_numpy(n, nc):
  """pcls_validation_update (csrc/validation.cu): focal / sparse-CE loss sums and the weighted confusion matrix in one
  pass, vs float64 numpy on the same float32 inputs; out-of-range labels / predictions (a zero one-hot row, a dropped
  pair), ragged sizes, absent mask / weights."""
  from pclsegmentation_b200 import _lib
  lib = _lib.load()
  rng = np.random.default_rng(n + nc)
  logits = rng.normal(0, 3, (n, nc)).astype(np.float32)
  e = np.exp(logits - logits.max(1, keepdims=True)) if n else logits
  probs = (e / e.sum(1, keepdims=True)).astype(np.float32) if n else logits
  label = rng.integers(0, nc, n).astype(np.int32)
  pred = rng.integers(0, nc, n).astype(np.int32)
  if n > 8:
    label[3], pred[5], label[7] = nc, -1, -2
  mask = (rng.random(n) < 0.7).astype(np.uint8)
  weight = rng.uniform(0.2, 3.0, n).astype(np.float32)
  eps, gamma = 1e-12, 2.0
  s = torch.cuda.current_stream().cuda_stream
  d = lambda a: torch.from_numpy(a).cuda()
  P, Y, Q, M, Wt = d(probs), d(label), d(pred), d(mask), d(weight)

  def run(kind, use_mask, use_w, with_cm):
    acc = torch.zeros(2, dtype=torch.float64, device="cuda")
    cm = torch.zeros((nc, nc), dtype=torch.float64, device="cuda") if with_cm else None
    dropped = torch.zeros(1, dtype=torch.int64, device="cuda")
    _lib.check(lib.pcls_validation_update(P.data_ptr(), Y.data_ptr(), Q.data_ptr() if with_cm else None,
                                          M.data_ptr() if use_mask else None, Wt.data_ptr() if use_w else None, n, nc, kind,
                                          eps, gamma, acc.data_ptr(), cm.data_ptr() if with_cm else None, dropped.data_ptr(),
                                          s), "pcls_validation_update")
    return acc.cpu().numpy(), None if cm is None else cm.cpu().numpy(), int(dropped.item())

  p64, w64 = probs.astype(np.float64), weight.astype(np.float64)
  ok_y = (label >= 0) & (label < nc)
  yc = np.where(ok_y, label, 0)
  rows = np.arange(n)
  for use_mask in (True, False):
    for use_w in (True, False):
      m = mask.astype(np.float64) if use_mask else np.ones(n)
      w = w64 if use_w else np.ones(n)
      # focal: p = float32(probs + eps) like the TF graph
      pe = (probs[rows, yc] + np.float32(eps)).astype(np.float64) if n else np.zeros(0)
      num = ((1.0 - pe) ** gamma * -np.log(pe) * w * m * ok_y).sum()
      acc, cm, dr = run(1, use_mask, use_w, True)
      assert abs(acc[0] - num) <= 2e-6 * max(1.0, abs(num)) and acc[1] == m.sum()
      okp = ok_y & (pred >= 0) & (pred < nc)
      ref = np.zeros((nc, nc))
      np.add.at(ref, (label[okp], pred[okp]), w[okp])
      assert np.allclose(cm, ref, rtol=1e-12, atol=1e-9) and dr == int((~okp).sum())
      # sparse CE
      pc = np.clip(p64, 1e-7, 1 - 1e-7)
      num = (-(np.log(pc[rows, yc]) - np.log(pc.sum(1))) * w * ok_y).sum() if n else 0.0
      acc, _, _ = run(2, False, use_w, False)
      assert abs(acc[0] - num) <= 2e-6 * max(1.0, abs(num)) and acc[1] == n
