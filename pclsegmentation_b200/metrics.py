"""``MeanIoU`` - the slice of ``tf.keras.metrics.MeanIoU`` the reference uses (eval.py:41,48,50,58;
nets/SegmentationNetwork.py:52): ``update_state(label, pred)``, ``total_cm``, ``result()``, ``reset_states()``.

The confusion matrix lives on the GPU as int64 (csrc/confusion.cu: shared-memory histogram kernel); TF keeps it in
float32, which is exact only below 2^24 per cell.  ``allreduce()`` is the one multi-GPU exchange step of the path:
one ncclAllReduce(int64, sum) over the per-GPU matrices.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .device import ptr, require_cuda, stream_handle, to_device


class MeanIoU:
  def __init__(self, num_classes, name="MeanIoU"):
    self.num_classes = int(num_classes)
    self.name = name
    self._cm = None
    self._cmw = None      # float64 matrix of weighted updates (test_step); None until the first weighted update
    self._dropped = None

  def _ensure(self):
    if self._cm is None:
      dev = require_cuda()
      self._cm = torch.zeros((self.num_classes, self.num_classes), dtype=torch.int64, device=dev)
      self._dropped = torch.zeros(1, dtype=torch.int64, device=dev)
    return self._cm

  def update_state(self, y_true, y_pred, sample_weight=None):
    """cm[label, pred] += 1 over every element (eval.py passes no weights: masked pixels count as None/None)."""
    cm = self._ensure()
    label = to_device(y_true, torch.int32).reshape(-1)
    pred = to_device(y_pred, torch.int32).reshape(-1)
    if label.numel() != pred.numel():
      raise ValueError("label and prediction sizes differ: %d vs %d" % (label.numel(), pred.numel()))
    if sample_weight is not None:
      # test_step (nets/SegmentationNetwork.py:129): tf.math.confusion_matrix(..., weights=w) sums the weights per cell
      # (float64 shared-memory histogram, csrc/validation.cu)
      w = to_device(sample_weight, torch.float32).reshape(-1)
      if w.numel() != label.numel():
        raise ValueError("weights and label sizes differ: %d vs %d" % (w.numel(), label.numel()))
      _lib.check(_lib.load().pcls_validation_update(None, ptr(label), ptr(pred), None, ptr(w), label.numel(),
                                                    self.num_classes, 0, 0.0, 0.0, None, ptr(self.weighted_cm()),
                                                    ptr(self._dropped), stream_handle()), "pcls_validation_update")
      return
    _lib.check(_lib.load().pcls_confusion_update(ptr(label), ptr(pred), label.numel(), self.num_classes, ptr(cm),
                                                 ptr(self._dropped), stream_handle()), "pcls_confusion_update")

  def weighted_cm(self):
    """The float64 [NC,NC] matrix of weighted updates (created on first use)."""
    cm = self._ensure()
    if self._cmw is None:
      self._cmw = torch.zeros((self.num_classes, self.num_classes), dtype=torch.float64, device=cm.device)
    return self._cmw

  @property
  def total_cm(self):
    """[NC,NC] CUDA tensor, rows = label, cols = prediction (tf.math.confusion_matrix layout): int64 counts, or
    float64 once weighted updates have been made."""
    cm = self._ensure()
    return cm if self._cmw is None else cm.to(torch.float64) + self._cmw

  @property
  def dropped(self):
    return int(self._dropped.item()) if self._dropped is not None else 0

  def allreduce(self, comm):
    """Sum the matrix over all ranks of ``comm`` (sharding.Communicator), in place, on the current stream: the int64
    counts with ONE ncclAllReduce through the C ABI; the float64 matrix of weighted updates (test_step) and the dropped
    counter, when present on any rank, with ``torch.distributed`` (off the hot path)."""
    comm.allreduce_confusion(self._ensure())
    comm.allreduce_aux(self)

  def result(self):
    """Mean IoU over the classes whose denominator is non-zero (tf.keras.metrics.MeanIoU.result)."""
    cm = self.total_cm.cpu().numpy()
    tp = np.diag(cm).astype(np.float64)
    denom = (cm.sum(0) + cm.sum(1)).astype(np.float64) - tp
    valid = denom != 0
    if not valid.any():
      return np.float32(0.0)
    iou = np.zeros_like(tp)
    np.divide(tp, denom, out=iou, where=valid)
    return np.float32(iou.sum() / valid.sum())

  def reset_states(self):
    if self._cm is not None:
      self._cm.zero_()
      self._dropped.zero_()
    self._cmw = None

  reset_state = reset_states


class Reliability:
  """Reliability of confidences (Guo et al., ICML 2017): ``n_bins`` equal bins of [0, 1], per bin the number of counted
  elements, how many of them are correct and the sum of their confidences, accumulated on the GPU
  (pcls_reliability_update: int64 / int64 / float64, a shared-memory histogram per block).  An element counts when its
  label and prediction are class ids in [0, num_classes) and the label is not ``ignore_index``.  Pixels and points go
  through the same kernel."""

  def __init__(self, n_bins, num_classes):
    self.n_bins, self.num_classes = int(n_bins), int(num_classes)
    if not 1 <= self.n_bins <= 64:
      raise ValueError("n_bins must be in [1, 64], got %d" % self.n_bins)
    self.count = self.correct = self.conf = None

  def _ensure(self, dev=None):
    if self.count is None:
      dev = dev if dev is not None else require_cuda()
      self.count = torch.zeros(self.n_bins, dtype=torch.int64, device=dev)
      self.correct = torch.zeros(self.n_bins, dtype=torch.int64, device=dev)
      self.conf = torch.zeros(self.n_bins, dtype=torch.float64, device=dev)

  def update_state(self, conf, pred, label, ignore_index=-1):
    """conf float32, pred / label int32: CUDA tensors (or arrays) of one size."""
    self._ensure()
    c = to_device(conf, torch.float32).reshape(-1)
    p = to_device(pred, torch.int32).reshape(-1)
    y = to_device(label, torch.int32).reshape(-1)
    if not c.numel() == p.numel() == y.numel():
      raise ValueError("conf / pred / label sizes differ: %d, %d, %d" % (c.numel(), p.numel(), y.numel()))
    _lib.check(_lib.load().pcls_reliability_update(ptr(c), ptr(p), ptr(y), c.numel(), self.num_classes, int(ignore_index),
                                                   self.n_bins, ptr(self.count), ptr(self.correct), ptr(self.conf),
                                                   stream_handle()), "pcls_reliability_update")

  def allreduce(self, comm):
    """Sums the bins over the ranks of ``comm`` (torch.distributed, off the hot path)."""
    self._ensure()
    comm.allreduce_sums([self.count, self.correct, self.conf])

  def reset_states(self):
    if self.count is not None:
      self.count.zero_()
      self.correct.zero_()
      self.conf.zero_()

  def result(self):
    """dict(ece, mce, accuracy, mean_confidence, count (N), and per bin: bin_lo, bin_hi, bin_count, bin_accuracy,
    bin_confidence (0 for an empty bin)).  ECE = sum_b |correct_b - conf_b| / N; MCE = max over the non-empty bins of
    |accuracy_b - confidence_b|; all 0 when nothing was counted."""
    if self.count is None:
      cnt, cor, cs = np.zeros(self.n_bins, np.int64), np.zeros(self.n_bins, np.int64), np.zeros(self.n_bins)
    else:
      cnt, cor, cs = self.count.cpu().numpy(), self.correct.cpu().numpy(), self.conf.cpu().numpy()
    return reliability_scores(cnt, cor, cs)


class UncertaintyAUROC:
  """How well an uncertainty u in [0, 1] detects misclassified elements, as a binned AUROC: ``n_bins`` equal bins of u
  hold the number of elements and of correct ones (pcls_reliability_update with u as the "confidence", so pixels and
  points share the kernel and its counting rule).  AUROC = P(u_error > u_correct) over (error, correct) pairs, a pair in
  the same bin counted 1/2; 0.5 when there are no errors or nothing correct.  Two uncertainties are tracked: the
  normalised predictive entropy H and the normalised mutual information MI of MC dropout."""

  def __init__(self, num_classes, n_bins=64):
    self.entropy = Reliability(n_bins, num_classes)
    self.mutual_information = Reliability(n_bins, num_classes)

  def update_state(self, entropy, mutual_information, pred, label, ignore_index=-1):
    self.entropy.update_state(entropy, pred, label, ignore_index)
    self.mutual_information.update_state(mutual_information, pred, label, ignore_index)

  def allreduce(self, comm):
    self.entropy.allreduce(comm)
    self.mutual_information.allreduce(comm)

  def result(self):
    """dict(auroc_entropy, auroc_mi, count, errors, and the integer bins: entropy_count / entropy_correct / mi_count /
    mi_correct)."""
    out = {}
    for key, r in (("entropy", self.entropy), ("mi", self.mutual_information)):
      r._ensure()
      cnt, cor = r.count.cpu().numpy(), r.correct.cpu().numpy()
      out["auroc_" + key] = binned_auroc(cnt, cor)
      out[key + "_count"], out[key + "_correct"] = cnt, cor
    out["count"] = int(out["entropy_count"].sum())
    out["errors"] = int(out["entropy_count"].sum() - out["entropy_correct"].sum())
    return out


def binned_auroc(count, correct):
  """AUROC of u for detecting errors from its histogram (per bin: elements, correct ones); see UncertaintyAUROC."""
  count = np.asarray(count, np.float64)
  correct = np.asarray(correct, np.float64)
  err = count - correct
  n_err, n_ok = err.sum(), correct.sum()
  if n_err == 0 or n_ok == 0:
    return 0.5
  below_ok = np.concatenate([[0.0], np.cumsum(correct)[:-1]])
  return float((err * (below_ok + 0.5 * correct)).sum() / (n_err * n_ok))


def reliability_scores(count, correct, conf_sum):
  """The scores of ``Reliability.result`` from the three per-bin sums (host, float64)."""
  count = np.asarray(count, np.int64)
  correct = np.asarray(correct, np.int64)
  conf_sum = np.asarray(conf_sum, np.float64)
  nb = count.size
  n = int(count.sum())
  full = count > 0
  acc_b = np.divide(correct, count, out=np.zeros(nb), where=full)
  conf_b = np.divide(conf_sum, count, out=np.zeros(nb), where=full)
  edges = np.arange(nb + 1) / nb
  return dict(ece=float(np.abs(correct - conf_sum).sum() / n) if n else 0.0,
              mce=float(np.abs(acc_b - conf_b)[full].max()) if n else 0.0,
              accuracy=float(correct.sum() / n) if n else 0.0, mean_confidence=float(conf_sum.sum() / n) if n else 0.0,
              count=n, bin_lo=edges[:-1], bin_hi=edges[1:], bin_count=count, bin_accuracy=acc_b, bin_confidence=conf_b)


class PanopticQuality:
  """Panoptic quality over thing classes (Kirillov et al., "Panoptic Segmentation", CVPR 2019), point-wise per scan, on
  the host (numpy; the caller hands over only the points that can be in a segment).  The rules are this project's; parity
  with semantic-kitti-api's evaluation script is not claimed.

  Per scan (``update``):
  * points whose ground-truth class is ``ignore_class`` (the config's "None") are removed first;
  * a ground-truth segment is the set of points of a thing class with equal (class, instance id), instance id > 0; one
    with fewer than ``min_gt_points`` points is ignored: it counts as neither TP nor FN;
  * a predicted segment is the set of points of a thing class with equal (class, instance id), instance id > 0;
  * a predicted and a ground-truth segment of the same class match when their IoU is > 0.5 (strictly); a match with a
    counted ground-truth segment is a TP, an unmatched counted ground-truth segment a FN, an unmatched predicted segment
    a FP unless more than half of its points lie in ignored ground-truth segments of its class.
  ``result()``: per thing class PQ = sum(IoU of TPs) / (TP + FP / 2 + FN / 2), SQ = sum(IoU) / TP (0 without TPs),
  RQ = TP / (TP + FP / 2 + FN / 2), and their means over the classes with at least one counted segment."""

  def __init__(self, num_classes, thing_classes, ignore_class=None, min_gt_points=50):
    self.num_classes = int(num_classes)
    self.thing_classes = sorted(int(c) for c in thing_classes)
    self.ignore_class = -1 if ignore_class is None else int(ignore_class)
    self.min_gt_points = int(min_gt_points)
    self._thing = np.zeros(self.num_classes + 1, bool)      # the last entry: any id outside [0, num_classes)
    self._thing[self.thing_classes] = True
    self.reset_states()

  def reset_states(self):
    self.tp = np.zeros(self.num_classes, np.int64)
    self.fp = np.zeros(self.num_classes, np.int64)
    self.fn = np.zeros(self.num_classes, np.int64)
    self.iou_sum = np.zeros(self.num_classes, np.float64)

  def _segments(self, cls, inst):
    ok = self._thing[np.where((cls >= 0) & (cls < self.num_classes), cls, self.num_classes)] & (inst > 0)
    key = cls * (1 << 32) + inst
    seg = np.full(cls.shape[0], -1, np.int64)
    uniq, inv, size = np.unique(key[ok], return_inverse=True, return_counts=True)
    seg[ok] = inv.reshape(-1)
    return seg, uniq >> 32, size

  def update(self, gt_class, gt_inst, pred_class, pred_inst):
    """One scan: per point the ground-truth class and instance id, the predicted class and instance id (any integer
    arrays of one length)."""
    gc, gi, pc, pi = (np.asarray(a, np.int64).reshape(-1) for a in (gt_class, gt_inst, pred_class, pred_inst))
    keep = gc != self.ignore_class
    gc, gi, pc, pi = gc[keep], gi[keep], pc[keep], pi[keep]
    gseg, gcls, gsize = self._segments(gc, gi)
    pseg, pcls, psize = self._segments(pc, pi)
    both = (gseg >= 0) & (pseg >= 0) & (gc == pc)
    pair, inter = np.unique(gseg[both] * max(psize.size, 1) + pseg[both], return_counts=True)
    g, p = pair // max(psize.size, 1), pair % max(psize.size, 1)
    iou = inter / (gsize[g] + psize[p] - inter).astype(np.float64)
    counted = gsize >= self.min_gt_points
    tp = (iou > 0.5) & counted[g]
    matched_g = np.zeros(gsize.size, bool)
    matched_g[g[tp]] = True
    matched_p = np.zeros(psize.size, bool)
    matched_p[p[tp]] = True
    in_ignored = np.bincount(p[~counted[g]], weights=inter[~counted[g]], minlength=psize.size)
    fp = ~matched_p & ~(in_ignored > 0.5 * psize)
    np.add.at(self.tp, gcls[g[tp]], 1)
    np.add.at(self.iou_sum, gcls[g[tp]], iou[tp])
    np.add.at(self.fn, gcls[counted & ~matched_g], 1)
    np.add.at(self.fp, pcls[fp], 1)

  def result(self):
    """dict(classes, pq, sq, rq, tp, fp, fn: per thing class, counted: which have a counted segment, pq_mean, sq_mean,
    rq_mean over the counted classes, 0 if none)."""
    c = np.asarray(self.thing_classes, np.int64)
    tp, fp, fn, s = self.tp[c], self.fp[c], self.fn[c], self.iou_sum[c]
    den = tp + 0.5 * fp + 0.5 * fn
    counted = den > 0
    pq = np.divide(s, den, out=np.zeros(c.size), where=counted)
    rq = np.divide(tp.astype(np.float64), den, out=np.zeros(c.size), where=counted)
    sq = np.divide(s, tp.astype(np.float64), out=np.zeros(c.size), where=tp > 0)
    mean = (lambda v: float(v[counted].mean()) if counted.any() else 0.0)
    return dict(classes=c, pq=pq, sq=sq, rq=rq, tp=tp, fp=fp, fn=fn, counted=counted, pq_mean=mean(pq),
                sq_mean=mean(sq), rq_mean=mean(rq))
