"""Device-resident pipelines over the C-ABI kernels:

* ``ScanSegmenter``  raw scans -> spherical projection -> network forward -> labels (BASELINE config 4: the converter's
  per-scan loop dataset_convert/semantic_kitti.py:152-179 fused with inference.py:44-78; range images never leave HBM),
  optionally one label per point (pcls_point_labels: back-projection or the k-NN vote of ``KNN``) and an instance id
  per thing-class point (pcls_point_instances: connected components of ``Clustering``); with a ``tta.TTA`` the forward
  runs over mirrored / rotated views and their merged predictions feed the rest
* ``ScanEvaluator``  point-wise evaluation on raw scans: scans -> point labels -> confusion update per point, and
  panoptic quality (``metrics.PanopticQuality``) when instances are asked for, and the reliability of the per-point
  confidences with a ``calibration.Calibration``
* ``Evaluator``      the eval.py hot loop (eval.py:45-50): forward -> head -> confusion update per batch on this rank's
  shard of the frames, one all-reduce of the int64 matrix at the end, then IoU / recall / precision / mIoU; with a
  ``calibration.Calibration`` also the reliability of the confidences (ECE / MCE) and the NLL of a temperature grid.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .calibration import TemperatureNLL, check_tta, confidence as pixel_confidence, raw_mask
from .device import ptr, samples_to_device, stream_handle, to_device
from .laserscan import SphericalProjector
from .mc_dropout import check_exclusive, forward_mc
from .metrics import MeanIoU, PanopticQuality, Reliability, UncertaintyAUROC
from .sharding import Communicator, shard_range
from .tta import forward_tta
from .utils.util import confusion_matrix_to_iou_recall_precision


class KNN:
  """Parameters of the k-NN vote that turns range-image predictions into per-point labels (pcls_point_labels).  The
  defaults are the post-processing settings published with RangeNet++ (window 5, k 5, sigma 1, cutoff 1 m, the
  unlabeled class ignored); ``ignore_class="none"`` resolves to the config's "None" class, an int is taken as is (-1 =
  count every class).  The window weights are 1 - g / sum(g), g = exp(-(dx^2 + dy^2) / (2 sigma^2)), computed in float64
  and rounded once to float32."""

  def __init__(self, search=5, k=5, sigma=1.0, cutoff=1.0, ignore_class="none"):
    self.search, self.k, self.sigma, self.cutoff, self.ignore_class = int(search), int(k), float(sigma), float(cutoff), \
        ignore_class

  def weights(self):
    p = (self.search - 1) // 2
    dy, dx = np.mgrid[-p:p + 1, -p:p + 1].astype(np.float64)
    g = np.exp(-(dx * dx + dy * dy) / (2.0 * self.sigma ** 2))
    return (1.0 - g / g.sum()).reshape(-1).astype(np.float32)

  def ignore_index(self, mc):
    return mc.CLASSES.index("None") if self.ignore_class == "none" else int(self.ignore_class)


# Thing classes by name, for ``Clustering(thing_classes=None)``: SemanticKITTI's eight, and the ika / nuScenes configs'
# road users.
THING_CLASS_NAMES = ("car", "bicycle", "motorcycle", "truck", "other-vehicle", "person", "bicyclist", "motorcyclist",
                     "Person", "Two-wheeler", "TwoWheeler", "Car", "Truck", "Bus")


class Clustering:
  """Parameters of the instance clustering of thing-class points (pcls_point_instances): pixels of the same thing
  class within ``rows`` rows and ``cols`` columns of each other (a (2 rows + 1) x (2 cols + 1) window; columns wrap
  around the 360-degree seam with ``wrap``) join when their points are at most ``tau`` metres apart; components with
  fewer than ``min_points`` points get no id.  ``thing_classes`` is a list of class names or ids; None takes the
  classes of ``THING_CLASS_NAMES`` that the config has.  The defaults (0.5 m, a 3 x 5 window, 10 points) are a
  starting point: they have not been tuned against real scans."""

  def __init__(self, tau=0.5, rows=1, cols=2, min_points=10, wrap=True, thing_classes=None):
    self.tau, self.rows, self.cols, self.min_points, self.wrap = float(tau), int(rows), int(cols), int(min_points), \
        bool(wrap)
    self.thing_classes = thing_classes

  def thing_ids(self, mc):
    """The thing classes as sorted class ids of config ``mc``."""
    if self.thing_classes is None:
      ids = [i for i, n in enumerate(mc.CLASSES) if n in THING_CLASS_NAMES]
      if not ids:
        raise ValueError("no thing class of %s is in the config's classes; pass thing_classes" % (THING_CLASS_NAMES,))
      return ids
    ids = sorted({mc.CLASSES.index(c) if isinstance(c, str) else int(c) for c in self.thing_classes})
    if ids and not 0 <= ids[0] <= ids[-1] < mc.NUM_CLASS:
      raise ValueError("thing class ids %s are not all in [0, %d)" % (ids, mc.NUM_CLASS))
    return ids

  def thing_mask(self, mc):
    return sum(1 << i for i in self.thing_ids(mc))


class ScanSegmenter:
  def __init__(self, model, fov_up=3.0, fov_down=-25.0, label_lut=None):
    mc = model.mc
    self.model, self.mc = model, mc
    self.projector = SphericalProjector(mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL, fov_up, fov_down, label_lut=label_lut)

  def segment_device(self, points, offsets, labels=None, want_probabilities=False, out=None, want_image=False,
                     want_logits=False, want_point_labels=False, knn=None, instances=None, tta=None, confidence=None,
                     mc_dropout=None):
    """points [total,4] float32 CUDA (x,y,z,remission), offsets [B+1] int64 CUDA -> dict(predictions, proj_idx,
    probabilities?, logits?, image?, point_labels?) - keys and activations stay on the device.

    Default (no image, no labels wanted): the resolve pass writes the NORMALISED 16-bit network input and the mask
    straight into the net's own buffers (pcls_project_resolve_net_input): no float32 [B,H,W,6] range image is written
    and read back, and the forward runs without its input kernel.  With want_image / labels the range image is
    materialised (the converters' output) and the forward reads it.

    want_point_labels: also one label per point, ``point_labels`` [total] int32 CUDA (pcls_point_labels on the same
    stream after the forward): with ``knn=None`` each point takes its pixel's prediction, with a ``KNN`` the k-NN vote
    decides; points the projection dropped get the "None" class.

    instances: a ``Clustering`` - also ``instances`` [total] int32 (0 = no instance, ids 1, 2, ... per scan) and
    ``instance_counts`` [B] int32 CUDA (pcls_point_instances on the same stream after the point labels); needs
    want_point_labels.

    tta: a ``tta.TTA`` - the range image is materialised and goes through ``tta.forward_tta``; the merged predictions
    (and probabilities) take the place of the forward's, and the point labels / instances are computed from them as
    they are.  Logits are not merged, so want_logits is refused with it.

    confidence: a temperature T - also ``confidence`` [B,H,W] float32 (max softmax(logits / T) per pixel, 0 at empty
    pixels; pcls_confidence) and ``point_confidence`` [total] float32 (the probability at T that the point's own pixel
    gives the point's label; pcls_point_confidence); needs want_point_labels.  At T = 1 the forward's probabilities are
    used as they are; with a TTA only T = 1 is available (the merged probabilities).

    mc_dropout: an ``mc_dropout.MCDropout`` - the range image is materialised and goes through
    ``mc_dropout.forward_mc``; the MC mean's predictions (and probabilities) take the place of the forward's, and the
    result also holds ``confidence`` / ``entropy`` / ``mutual_information`` [B,H,W] and, with want_point_labels,
    ``point_mi`` / ``point_entropy`` [total] float32 (the value of the point's own pixel, 0 for a dropped point) and
    ``point_confidence``: as with ``confidence=1``, the MC mean's probability of the label the point got.  Refused with a
    TTA, logits or a temperature other than 1."""
    if mc_dropout is not None and (tta is not None or want_logits or (confidence is not None and
                                                                      float(confidence) != 1.0)):
      raise ValueError("MC dropout cannot be combined with test-time augmentation, logits or a softmax temperature")
    if mc_dropout is not None and want_point_labels:
      confidence = 1.0     # one definition of the point confidence under MC: the mean's probability of the point's label
    if instances is not None and not want_point_labels:
      raise ValueError("instances need the point labels: segment with want_point_labels=True")
    if tta is not None and want_logits:
      raise ValueError("test-time augmentation merges probabilities, not logits: segment without want_logits")
    if confidence is not None:
      if not want_point_labels:
        raise ValueError("confidence needs the point labels: segment with want_point_labels=True")
      if tta is not None and float(confidence) != 1.0:
        raise ValueError("test-time augmentation merges probabilities, not logits: confidence with TTA is only "
                         "available at temperature 1")
    tempered = confidence is not None and float(confidence) != 1.0
    fwd_probs = want_probabilities or (confidence is not None and not tempered)
    fwd_logits = want_logits or tempered
    B = int(offsets.numel()) - 1
    if mc_dropout is not None or tta is not None or want_image or labels is not None or B > self._staged_capacity(B):
      proj = self.projector.project(points, offsets, labels=labels, empty_fill=0.0, want_point_outputs=want_point_labels)
      if mc_dropout is not None:
        res = forward_mc(self.model, proj["image"], mc_dropout, want_probabilities=fwd_probs, out=out)
        if want_point_labels:
          for k, name in (("mutual_information", "point_mi"), ("entropy", "point_entropy")):
            res[name] = self._point_gather(res[k], offsets, proj["proj_x"], proj["proj_y"])
      elif tta is not None:
        res = forward_tta(self.model, proj["image"], tta, want_probabilities=fwd_probs, out=out)
      else:
        res = self.model.forward_device(proj["image"], None, mean=self.mc.INPUT_MEAN, std=self.mc.INPUT_STD,
                                        want_probabilities=fwd_probs, want_logits=fwd_logits, out=out)
      res.update(image=proj["image"], proj_idx=proj["proj_idx"])
      if want_point_labels:
        res["point_labels"] = self._point_labels(res["predictions"], proj["keys"], offsets, proj["proj_x"],
                                                 proj["proj_y"], proj["unproj_range"], knn)
        if instances is not None:
          res.update(self._instances(points, proj["keys"], offsets, proj["proj_x"], proj["proj_y"],
                                     res["point_labels"], instances))
        if confidence is not None:
          res.update(self._confidence(res, raw_mask(proj["image"], self.mc), offsets, proj["proj_x"], proj["proj_y"],
                                      float(confidence), want_probabilities, want_logits))
      return res
    lib = _lib.load()
    H, W = self.projector.H, self.projector.W
    inp, msk, _ = self.model.input_buffers(B)
    keys = torch.empty((B, H, W), dtype=torch.int64, device=points.device)
    idx = torch.empty((B, H, W), dtype=torch.int32, device=points.device)
    px = py = ur = None
    if want_point_labels:
      total = int(points.shape[0])
      px = torch.empty(total, dtype=torch.int32, device=points.device)
      py = torch.empty(total, dtype=torch.int32, device=points.device)
      ur = torch.empty(total, dtype=torch.float32, device=points.device)
    s = stream_handle()
    _lib.check(lib.pcls_project_scatter(ptr(points), None, ptr(offsets), B, int(points.shape[0]), H, W,
                                        float(self.projector.fov_up), float(self.projector.fov_down), ptr(keys), ptr(px),
                                        ptr(py), ptr(ur), s), "pcls_project_scatter")
    mean = (ctypes.c_double * 5)(*np.asarray(self.mc.INPUT_MEAN, np.float64).reshape(-1))
    std = (ctypes.c_double * 5)(*np.asarray(self.mc.INPUT_STD, np.float64).reshape(-1))
    _lib.check(lib.pcls_project_resolve_net_input(ptr(points), ptr(offsets), B, H, W, ptr(keys), mean, std,
                                                  self.model.precision, inp, msk, ptr(idx), s),
               "pcls_project_resolve_net_input")
    res = self.model.forward_staged(B, want_probabilities=fwd_probs, want_logits=fwd_logits, out=out)
    res.update(proj_idx=idx)
    if want_point_labels:
      res["point_labels"] = self._point_labels(res["predictions"], keys, offsets, px, py, ur, knn)
      if instances is not None:
        res.update(self._instances(points, keys, offsets, px, py, res["point_labels"], instances))
      if confidence is not None:
        # the net's own mask buffer holds this batch's mask (range > 0) until the next forward
        res.update(self._confidence(res, msk, offsets, px, py, float(confidence), want_probabilities, want_logits))
    return res

  def _confidence(self, res, mask, offsets, px, py, T, want_probabilities, want_logits):
    """Pixel confidence at temperature T and the per-point confidence of the point labels; drops the probabilities /
    logits the caller did not ask for."""
    nc = self.mc.NUM_CLASS
    if T != 1.0:
      c = pixel_confidence(nc, logits=res["logits"], mask=mask, temperature=T, want_probs=True)
      probs = c["probabilities"]
    else:
      probs = res["probabilities"]
      c = pixel_confidence(nc, probs=probs, mask=mask)
    B, H, W = res["predictions"].shape
    total = int(px.numel())
    pc = torch.empty(total, dtype=torch.float32, device=probs.device)
    _lib.check(_lib.load().pcls_point_confidence(ptr(probs), ptr(offsets), B, H, W, total, ptr(px), ptr(py),
                                                 ptr(res["point_labels"]), nc, ptr(pc), stream_handle()),
               "pcls_point_confidence")
    if not want_probabilities:
      res.pop("probabilities", None)
    if not want_logits:
      res.pop("logits", None)
    return dict(confidence=c["confidence"], point_confidence=pc)

  def _point_gather(self, values, offsets, px, py):
    """values [B,H,W] float32 -> [total] float32: each point's own pixel's value, 0 for a dropped point (the exact
    gather of pcls_point_confidence with one class and every label 0)."""
    B, H, W = values.shape
    total = int(px.numel())
    zero = torch.zeros(total, dtype=torch.int32, device=values.device)
    out = torch.empty(total, dtype=torch.float32, device=values.device)
    _lib.check(_lib.load().pcls_point_confidence(ptr(values.contiguous()), ptr(offsets), B, H, W, total, ptr(px),
                                                 ptr(py), ptr(zero), 1, ptr(out), stream_handle()),
               "pcls_point_confidence")
    return out

  def _point_labels(self, preds, keys, offsets, px, py, ur, knn):
    B, H, W = preds.shape
    total = int(px.numel())
    out = torch.empty(total, dtype=torch.int32, device=preds.device)
    search, k, w, cutoff, ignore, scratch = 1, 1, None, 0.0, -1, None
    if knn is not None:
      search, k, cutoff, ignore = knn.search, knn.k, knn.cutoff, knn.ignore_index(self.mc)
      wt = knn.weights()
      w = (ctypes.c_float * wt.size)(*wt.tolist())
      if search > 1:
        scratch = torch.empty((B, H, W), dtype=torch.int64, device=preds.device)
    _lib.check(_lib.load().pcls_point_labels(ptr(preds), ptr(keys), ptr(offsets), B, H, W, total, ptr(px), ptr(py),
                                             ptr(ur), self.mc.NUM_CLASS, self.mc.CLASSES.index("None"), search, k, w,
                                             float(cutoff), ignore, ptr(scratch), ptr(out), stream_handle()),
               "pcls_point_labels")
    return out

  def _instances(self, points, keys, offsets, px, py, labels, clustering):
    B, H, W = keys.shape
    total = int(px.numel())
    dev = keys.device
    lib = _lib.load()
    nbytes = _lib.check(lib.pcls_point_instances_scratch_bytes(B, H, W), "pcls_point_instances_scratch_bytes")
    scratch = torch.empty(max(nbytes // 4, 4), dtype=torch.float32, device=dev)   # allocations are 256-byte aligned
    inst = torch.empty(total, dtype=torch.int32, device=dev)
    counts = torch.empty(B, dtype=torch.int32, device=dev)
    _lib.check(lib.pcls_point_instances(ptr(points), ptr(keys), ptr(offsets), B, H, W, total, ptr(px), ptr(py),
                                        ptr(labels), self.mc.NUM_CLASS, clustering.thing_mask(self.mc),
                                        clustering.rows, clustering.cols, int(clustering.wrap), clustering.tau,
                                        clustering.min_points, ptr(scratch), ptr(inst), ptr(counts), stream_handle()),
               "pcls_point_instances")
    return dict(instances=inst, instance_counts=counts)

  def _staged_capacity(self, B):
    return self.model.input_buffers(B)[2]

  def segment(self, scans, labels=None, **kw):
    """scans: list of [N_i,4] float32 numpy arrays."""
    lens = [int(s.shape[0]) for s in scans]
    dev = self.projector._dev
    offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)).to(dev)
    pts = to_device(np.concatenate(scans, axis=0), torch.float32)
    lab = None
    if labels is not None:
      lab = to_device(np.concatenate(labels).astype(np.uint32).view(np.int32), torch.int32)
    kw.setdefault("want_image", True)     # host convenience: the projected range images come back with the labels
    return self.segment_device(pts, offsets, labels=lab, **kw)

  def point_labels(self, res, points_per_scan):
    """The ``point_labels`` of a ``segment_device(..., want_point_labels=True)`` result as one int32 numpy array per
    scan (lengths ``points_per_scan``)."""
    if "point_labels" not in res:
      raise ValueError("the result holds no point labels: segment with want_point_labels=True")
    lab = res["point_labels"].cpu().numpy()
    sizes = [int(n) for n in points_per_scan]
    if sum(sizes) != lab.shape[0]:
      raise ValueError("points_per_scan sums to %d, the result has %d point labels" % (sum(sizes), lab.shape[0]))
    return np.split(lab, np.cumsum(sizes)[:-1])

  def label_words(self, res, points_per_scan, inv_lut=None):
    """SemanticKITTI ``.label`` words of a result, one uint32 numpy array per scan: ``(instance << 16) | sem`` with sem
    = ``inv_lut[label]`` (e.g. the yaml's learning_map_inv as a LUT) or the class id, instance 0 when the result holds
    no ``instances``.  Raises if an id does not fit in 16 bits."""
    sems = self.point_labels(res, points_per_scan)
    words = [(inv_lut[s] if inv_lut is not None else s).astype(np.uint32) for s in sems]
    if any(int(w.max(initial=0)) > 0xFFFF for w in words):
      raise ValueError("a semantic id does not fit in the lower 16 bits of a label word")
    if "instances" not in res:
      return words
    inst = res["instances"].cpu().numpy()
    if int(inst.max(initial=0)) > 0xFFFF:
      raise ValueError("instance id %d does not fit in the upper 16 bits of a label word" % int(inst.max()))
    parts = np.split(inst.astype(np.uint32), np.cumsum([int(n) for n in points_per_scan])[:-1])
    return [(i << np.uint32(16)) | w for i, w in zip(parts, words)]


class Evaluator:
  """eval.py:33-58 on one rank; ``comm`` sums the confusion matrix over ranks (sharding.Communicator) or is None.
  ``tta``: a ``tta.TTA`` - the predictions are merged over its views (``tta.forward_tta``).
  ``calibration``: a ``calibration.Calibration`` - the forward also returns its logits; the confidence at the
  calibration's temperature (pcls_confidence) is binned against the head's predictions and the fixed-up labels, the
  "None" class ignored (``metrics.Reliability``), and the NLL at T = 1, at the temperature and, with ``fit``, on the
  grid is accumulated (``calibration.TemperatureNLL``).  With a TTA the merged probabilities give the confidence, so
  only T = 1 without a fit is available.
  ``mc_dropout``: an ``mc_dropout.MCDropout`` - the predictions are the MC mean's (``mc_dropout.forward_mc``), and the
  AUROC of H and of MI for detecting misclassified pixels (``metrics.UncertaintyAUROC``) and the reliability of the
  mean's confidence are accumulated, the "None" class ignored; refused with a TTA or a temperature / fit."""

  def __init__(self, model, comm=None, tta=None, calibration=None, mc_dropout=None):
    check_tta(calibration, tta)
    check_exclusive(mc_dropout, tta, calibration)
    self.model, self.mc = model, model.mc
    self.comm, self.tta, self.calibration, self.mc_dropout = comm, tta, calibration, mc_dropout
    self.miou_tracker = MeanIoU(num_classes=self.mc.NUM_CLASS, name="MeanIoU")
    self._none = self.mc.CLASSES.index("None")
    self.reliability = self.nll = self.auroc = self.mc_reliability = None
    if mc_dropout is not None:
      self.auroc = UncertaintyAUROC(self.mc.NUM_CLASS)
      self.mc_reliability = Reliability(calibration.n_bins if calibration is not None else 15, self.mc.NUM_CLASS)
    if calibration is not None:
      self.reliability = Reliability(calibration.n_bins, self.mc.NUM_CLASS)
      if tta is None and mc_dropout is None:
        self.nll = TemperatureNLL(calibration, self.mc.NUM_CLASS, self._none)
    self._mean = (ctypes.c_double * 5)(*np.asarray(self.mc.INPUT_MEAN).reshape(-1))
    self._std = (ctypes.c_double * 5)(*np.asarray(self.mc.INPUT_STD).reshape(-1))

  def update(self, samples, return_label=False):
    """samples: [B,H,W,6] float64 / float32 (x,y,z,i,d,label) numpy or CUDA tensor - the .npy frames of the dataset.
    Runs the fused input stage + forward + head, fixes the labels up (label[~mask] = None, data_loader.py:176) and
    accumulates the confusion matrix; nothing returns to the host."""
    x = samples_to_device(samples)
    B, H, W, C = x.shape
    if C != 6:
      raise ValueError("evaluation samples need 6 channels (x,y,z,intensity,depth,label)")
    cal = self.calibration is not None
    if self.mc_dropout is not None:
      res = forward_mc(self.model, x, self.mc_dropout)
    elif self.tta is not None:
      res = forward_tta(self.model, x, self.tta, want_probabilities=cal)
    else:
      res = self.model.forward_device(x, None, mean=self.mc.INPUT_MEAN, std=self.mc.INPUT_STD, want_probabilities=False,
                                      want_logits=cal)
    label = torch.empty((B, H, W), dtype=torch.int32, device=x.device)
    _lib.check(_lib.load().pcls_input_stage(ptr(x), 6, B * H * W, self._mean, self._std, self._none, None, None,
                                            ptr(label), None, 0, None, stream_handle()), "pcls_input_stage")
    self.miou_tracker.update_state(label, res["predictions"])
    if self.mc_dropout is not None:
      # masked pixels carry the "None" label after the fix-up, so they are not binned
      self.auroc.update_state(res["entropy"], res["mutual_information"], res["predictions"], label, self._none)
      self.mc_reliability.update_state(res["confidence"], res["predictions"], label, self._none)
      if cal:
        self.reliability.update_state(res["confidence"], res["predictions"], label, self._none)
    elif cal:
      nc = self.mc.NUM_CLASS
      if self.tta is not None:
        conf = pixel_confidence(nc, probs=res["probabilities"])["confidence"]
      else:
        conf = pixel_confidence(nc, logits=res["logits"], temperature=self.calibration.temperature)["confidence"]
        self.nll.update(res["logits"], label)
      # masked pixels carry the "None" label after the fix-up, so they are not binned
      self.reliability.update_state(conf, res["predictions"], label, self._none)
    return (res["predictions"], label) if return_label else res["predictions"]

  def finish(self):
    """All-reduce (if sharded) and compute the report of eval.py:50-58."""
    if self.comm is not None:
      self.miou_tracker.allreduce(self.comm)
    cm = self.miou_tracker.total_cm
    iou, recall, precision = confusion_matrix_to_iou_recall_precision(cm)
    rep = dict(confusion_matrix=cm.cpu().numpy(), iou=iou, recall=recall, precision=precision,
               miou=float(self.miou_tracker.result()))
    if self.calibration is not None:
      nll = self.nll if self.mc_dropout is None else None
      rep["calibration"] = _calibration_report(self.calibration, self.reliability, nll, self.comm)
    if self.mc_dropout is not None:
      rep["mc_dropout"] = _mc_report(self.mc_dropout, self.mc, self.auroc, self.mc_reliability, self.comm)
    return rep


def _mc_report(mcd, mc, auroc, reliability, comm):
  """dict(passes, rate, seed, uncertainty: ``UncertaintyAUROC.result()``, reliability: ``Reliability.result()`` of the
  MC mean's confidence), the sums all-reduced first when ``comm`` is given."""
  if comm is not None:
    auroc.allreduce(comm)
    reliability.allreduce(comm)
  return dict(passes=mcd.passes, rate=mcd.rate_for(mc), seed=mcd.seed, uncertainty=auroc.result(),
              reliability=reliability.result())


def _calibration_report(calibration, reliability, nll, comm):
  """dict(temperature, n_bins, reliability: ``Reliability.result()``, nll: ``TemperatureNLL.result()`` or None), the
  sums all-reduced first when ``comm`` is given."""
  if comm is not None:
    reliability.allreduce(comm)
    if nll is not None:
      nll.allreduce(comm)
  return dict(temperature=calibration.temperature, n_bins=calibration.n_bins, reliability=reliability.result(),
              nll=nll.result() if nll is not None else None)


class ScanEvaluator:
  """Point-wise evaluation on raw scans (single GPU): per batch projection -> forward -> per-point labels (``knn``:
  a ``KNN`` or None for the plain back-projection) -> ground truth ``label_lut[word & 0xFFFF]`` (pcls_map_labels; the raw
  semantic id without a LUT) -> confusion update over the points.  ``finish()`` gives the report of
  ``Evaluator.finish``.  With ``instances`` (a ``Clustering``) each batch also gets instance ids and feeds a
  ``PanopticQuality`` whose ground-truth instance id is the upper half of the label word (``word >> 16``); only the
  points in a predicted or ground-truth thing segment come back to the host.  ``tta``: a ``tta.TTA`` for the forward
  (``ScanSegmenter.segment_device(tta=)``).  ``calibration``: a ``calibration.Calibration`` without ``fit`` (the
  temperature is fitted on pixels, with ``Evaluator``) - each point's confidence at its temperature
  (``segment_device(confidence=)``) is binned against its label and the ground truth, the "None" class ignored.
  ``mc_dropout``: an ``mc_dropout.MCDropout`` - the point labels come from the MC mean, and the AUROC of each point's H
  and MI (its own pixel's) for detecting misclassified points and the reliability of the MC confidence are accumulated."""

  def __init__(self, model, fov_up=3.0, fov_down=-25.0, label_lut=None, knn=None, instances=None, tta=None,
               calibration=None, mc_dropout=None):
    check_tta(calibration, tta)
    check_exclusive(mc_dropout, tta, calibration)
    if calibration is not None and calibration.fit:
      raise ValueError("the temperature is fitted on pixels (Evaluator); point-wise evaluation takes a fixed temperature")
    self.seg = ScanSegmenter(model, fov_up, fov_down)
    self.mc, self.knn, self.instances, self.tta = model.mc, knn, instances, tta
    self.calibration, self.mc_dropout = calibration, mc_dropout
    self.reliability = Reliability(calibration.n_bins, self.mc.NUM_CLASS) if calibration is not None else None
    self.auroc = self.mc_reliability = None
    if mc_dropout is not None:
      self.auroc = UncertaintyAUROC(self.mc.NUM_CLASS)
      self.mc_reliability = Reliability(calibration.n_bins if calibration is not None else 15, self.mc.NUM_CLASS)
    self.miou_tracker = MeanIoU(num_classes=self.mc.NUM_CLASS, name="MeanIoU")
    self.pq = None
    if instances is not None:
      self.pq = PanopticQuality(self.mc.NUM_CLASS, instances.thing_ids(self.mc), self.mc.CLASSES.index("None"))
    self.lut = None
    if label_lut is not None:
      self.lut = torch.as_tensor(np.asarray(label_lut, dtype=np.int32)).to(self.seg.projector._dev)

  def update(self, batch):
    """batch: the dict ``dataset_convert.ScanBatchLoader.load`` returns, with labels.  Returns the segment_device result
    (``point_labels`` included) and the per-point ground truth ``gt`` [total] int32 CUDA."""
    if batch.get("labels") is None:
      raise ValueError("point-wise evaluation needs the label files")
    res = self.seg.segment_device(batch["points"], batch["offsets"], want_point_labels=True, knn=self.knn,
                                  instances=self.instances, tta=self.tta,
                                  confidence=self.calibration.temperature if self.calibration is not None else None,
                                  mc_dropout=self.mc_dropout)
    gt = self.ground_truth(batch)
    self.miou_tracker.update_state(gt, res["point_labels"])
    if self.reliability is not None:
      self.reliability.update_state(res["point_confidence"], res["point_labels"], gt, self.mc.CLASSES.index("None"))
    if self.auroc is not None:
      none = self.mc.CLASSES.index("None")
      self.auroc.update_state(res["point_entropy"], res["point_mi"], res["point_labels"], gt, none)
      self.mc_reliability.update_state(res["point_confidence"], res["point_labels"], gt, none)
    res["gt"] = gt
    if self.pq is not None:
      self._update_pq(batch, gt, res)
    return res

  def ground_truth(self, batch):
    """The per-point ground truth of a batch with labels: [total] int32 CUDA, ``label_lut[word & 0xFFFF]``."""
    n = int(batch["points"].shape[0])
    gt = torch.empty(n, dtype=torch.int32, device=batch["points"].device)
    lut = self.lut
    _lib.check(_lib.load().pcls_map_labels(ptr(batch["labels"]), n, ptr(lut), int(lut.numel()) if lut is not None else 0,
                                           ptr(gt), stream_handle()), "pcls_map_labels")
    return gt

  def _update_pq(self, batch, gt, res):
    """Feeds ``self.pq`` scan by scan with the points that can be in a segment: a predicted instance, or a ground-truth
    thing point with an instance id; points of the "None" class are left out (the metric removes them anyway)."""
    dev = gt.device
    gt_inst = (batch["labels"] >> 16) & 0xFFFF
    thing = torch.zeros(self.mc.NUM_CLASS + 1, dtype=torch.bool, device=dev)
    thing[torch.as_tensor(self.pq.thing_classes, dtype=torch.long, device=dev)] = True
    gcls = torch.where((gt >= 0) & (gt < self.mc.NUM_CLASS), gt, self.mc.NUM_CLASS).long()
    keep = (gt != self.pq.ignore_class) & ((res["instances"] > 0) | (thing[gcls] & (gt_inst > 0)))
    sizes = torch.as_tensor(batch["sizes"], dtype=torch.long, device=dev)
    scan = torch.repeat_interleave(torch.arange(len(batch["sizes"]), device=dev), sizes)
    cols = [t[keep].cpu().numpy() for t in (scan, gt, gt_inst, res["point_labels"], res["instances"])]
    bounds = np.searchsorted(cols[0], np.arange(len(batch["sizes"]) + 1))
    for b in range(len(batch["sizes"])):
      sl = slice(bounds[b], bounds[b + 1])
      self.pq.update(cols[1][sl], cols[2][sl], cols[3][sl], cols[4][sl])

  def finish(self):
    """The report of ``Evaluator.finish`` plus ``dropped``: points whose ground truth is not a class id (a raw semantic
    id with no LUT, e.g. KITTI's 10 / 40 / 252); they are not in the matrix.  With instances, also ``panoptic``: the
    ``PanopticQuality.result()`` report."""
    cm = self.miou_tracker.total_cm
    iou, recall, precision = confusion_matrix_to_iou_recall_precision(cm)
    rep = dict(confusion_matrix=cm.cpu().numpy(), iou=iou, recall=recall, precision=precision,
               miou=float(self.miou_tracker.result()), dropped=self.miou_tracker.dropped)
    if self.pq is not None:
      rep["panoptic"] = self.pq.result()
    if self.calibration is not None:
      rep["calibration"] = _calibration_report(self.calibration, self.reliability, None, None)
    if self.mc_dropout is not None:
      rep["mc_dropout"] = _mc_report(self.mc_dropout, self.mc, self.auroc, self.mc_reliability, None)
    return rep


def shard_files(files, comm=None):
  files = sorted(files)
  if comm is None or comm.world_size == 1:
    return files
  lo, hi = shard_range(len(files), comm.rank, comm.world_size)
  return files[lo:hi]
