"""``PCLSegmentationNetwork`` - base class of the segmentation networks.

Mirrors pcl_segmentation/nets/SegmentationNetwork.py: the constructor fields (:31-53), the ``call`` contract
``model([lidar_input, lidar_mask]) -> (probabilities, predictions)`` (:55-69), ``predict_step`` (:133-136), the
``miou_tracker`` and ``get_config`` (:144-151).  The forward itself - the traced layer graph plus ``segmentation_head``
(softmax -> argmax -> depth-zero mask, :58-69) - runs in libpclseg (pcls_net_forward).  ``test_step`` (:118-131) with
both losses (:71-91, :49) and the weighted MeanIoU is provided forward-only; ``train_step`` and the optimizer are out of
scope of this inference path.
"""
import ctypes

import numpy as np
import torch

from .. import _lib
from ..device import DeviceTensor, ptr, require_cuda, stream_handle, to_device, wrap
from ..metrics import MeanIoU
from .layers import Graph


def _dev(x, dtype):
  """host array / CUDA tensor (incl. the DeviceTensor wrappers the forward returns) -> plain CUDA tensor of `dtype`."""
  if torch.is_tensor(x) and x.is_cuda:
    return x.detach().as_subclass(torch.Tensor).to(dtype)
  return to_device(x, dtype)


class PCLSegmentationNetwork:
  """Base Class for segmentation networks (inference path)."""

  def __init__(self, mc):
    self.mc = mc
    self.NUM_CLASS = mc.NUM_CLASS
    self.BATCH_SIZE = mc.BATCH_SIZE
    self.ZENITH_LEVEL = mc.ZENITH_LEVEL
    self.AZIMUTH_LEVEL = mc.AZIMUTH_LEVEL
    self.NUM_FEATURES = mc.NUM_FEATURES
    self.CLASSES = mc.CLASSES
    self.CLS_COLOR_MAP = mc.CLS_COLOR_MAP
    assert self.NUM_FEATURES == 6, "the path implements the reference's 6-channel input (5 lidar channels + mask)"

    self.miou_tracker = MeanIoU(num_classes=self.NUM_CLASS, name="MeanIoU")
    self._loss_sum, self._loss_count = 0.0, 0          # loss_tracker = tf.keras.metrics.Mean (:53)

    self.precision = _lib.PCLS_F16
    self.net_options = {}
    self._graph = Graph(self.ZENITH_LEVEL, self.AZIMUTH_LEVEL)
    self._logits_sym = None
    self._taps = {}          # name -> symbolic tensor, recorded by call() (per-layer parity tests, see read_tap)
    self._net = None
    self._net_batch = 0
    self._mc_nets = {}       # dropout rate -> (stochastic pcls_net handle, its batch capacity); see mc_net
    self._pinned = {}

  # ---- the subclass provides call(); tracing it builds the op program and creates the variables ----
  def call(self, inputs, training=False, mask=None):
    raise NotImplementedError("Method should be called in child class!")

  def _trace(self):
    self._logits_sym = self.call([self._graph.input, None])

  def _tap(self, name, x):
    """Names an intermediate tensor of call() (same names as the `taps` of oracle/nn.py)."""
    self._taps[name] = x
    return x

  def read_tap(self, name, batch, net=None):
    """float32 CUDA copy [batch,H,width,channels] of a tapped intermediate of the LAST forward (of ``net``, e.g. an
    ``mc_net`` handle; default: the default net).  Intermediates share a liveness-planned arena, so this is only
    meaningful with set_option("keep_tensors", 1)."""
    if not self.net_options.get("keep_tensors"):
      raise _lib.PclsError("read_tap needs set_option('keep_tensors', 1) before the forward")
    sym = self._taps[name]
    out = torch.empty((batch, self.ZENITH_LEVEL, sym.width, sym.channels), dtype=torch.float32,
                      device=torch.device("cuda", torch.cuda.current_device()))
    _lib.check(_lib.load().pcls_net_read_tensor(self._net if net is None else net, sym.tid, batch, ptr(out),
                                                stream_handle()),
               "pcls_net_read_tensor")
    return out

  def segmentation_head(self, logits, lidar_mask):
    """Symbolic marker: the head (softmax, argmax, mask fill with CLASSES.index("None")) is executed by
    pcls_net_forward on the tensor returned here."""
    return logits

  # ---- variables (Keras attribute paths) -----------------------------------------------------------
  @property
  def variables(self):
    return self._graph.variables

  def get_weights_dict(self):
    return {k: v.copy() for k, v in self._graph.variables.items()}

  def set_weights_dict(self, weights, strict=True):
    """weights: {keras attribute path: array}; also accepts TF checkpoint style keys ending in
    '/.ATTRIBUTES/VARIABLE_VALUE'."""
    seen = set()
    for k, v in weights.items():
      k = k.replace("/.ATTRIBUTES/VARIABLE_VALUE", "")
      if k not in self._graph.variables:
        if strict and not k.startswith(("miou_tracker", "loss_tracker", "optimizer")):
          raise KeyError("unknown variable %r" % k)
        continue
      v = np.asarray(v, dtype=np.float32)
      if v.shape != self._graph.variables[k].shape:
        raise ValueError("variable %r has shape %s, expected %s" % (k, v.shape, self._graph.variables[k].shape))
      self._graph.variables[k] = v.copy()
      seen.add(k)
    if strict and len(seen) != len(self._graph.variables):
      raise KeyError("missing variables: %s" % sorted(set(self._graph.variables) - seen)[:5])
    self._release()

  def save_weights_npz(self, path):
    np.savez(path, **self._graph.variables)

  def load_weights_npz(self, path):
    with np.load(path) as f:
      self.set_weights_dict({k: f[k] for k in f.files})

  def load_weights(self, path):
    """`--path_to_model` of inference.py:128 / eval.py:73.  Accepts what the reference's training writes - a Keras
    SavedModel directory (`train.py:60`) or a checkpoint prefix (`train.py:42`), read without TensorFlow by
    utils/tensor_bundle.py - or the neutral `.npz` container keyed by Keras attribute paths.  Every variable of the
    network must be present (metrics / optimizer entries of the checkpoint are ignored)."""
    if str(path).endswith(".npz"):
      return self.load_weights_npz(path)
    from ..utils import tensor_bundle
    found = tensor_bundle.load_keras_variables(path)
    mine = {k: v for k, v in found.items() if k in self._graph.variables}
    missing = sorted(set(self._graph.variables) - set(mine))
    if missing:
      raise KeyError("%s: %d of %d network variables are missing (first: %s); the checkpoint holds %d variables, e.g. %s"
                     % (path, len(missing), len(self._graph.variables), missing[:3], len(found), sorted(found)[:3]))
    self.set_weights_dict(mine)

  def save_weights_bundle(self, prefix):
    """Writes the variables as a TensorBundle (checkpoint prefix) under their Keras object-graph keys."""
    from ..utils import tensor_bundle
    tensor_bundle.write_bundle(prefix, {k + "/.ATTRIBUTES/VARIABLE_VALUE": v for k, v in self._graph.variables.items()})

  def randomize_batch_norm(self, seed=0):
    """Random BN statistics / affine (mu ~ N(0,0.1), var ~ U(0.5,1.5), gamma ~ U(0.8,1.2), beta ~ N(0,0.1)) so that
    the BN folding is exercised (SURVEY.md §8d config 2); random biases ~ N(0, 0.05) likewise."""
    rng = np.random.default_rng(seed)
    for k in sorted(self._graph.variables):
      shape = self._graph.variables[k].shape
      if k.endswith("/moving_mean") or k.endswith("/beta"):
        self._graph.variables[k] = rng.normal(0, 0.1, shape).astype(np.float32)
      elif k.endswith("/moving_variance"):
        self._graph.variables[k] = rng.uniform(0.5, 1.5, shape).astype(np.float32)
      elif k.endswith("/gamma"):
        self._graph.variables[k] = rng.uniform(0.8, 1.2, shape).astype(np.float32)
      elif k.endswith("/bias"):
        self._graph.variables[k] = rng.normal(0, 0.05, shape).astype(np.float32)
    self._release()

  # ---- device execution ------------------------------------------------------------------------------
  def _release(self):
    if self._net is not None:
      _lib.load().pcls_net_destroy(self._net)
      self._net, self._net_batch = None, 0
    for handle, _ in self._mc_nets.values():
      _lib.load().pcls_net_destroy(handle)
    self._mc_nets.clear()

  def __del__(self):
    try:
      self._release()
    except Exception:
      pass

  def set_option(self, name, value):
    """Execution knobs of the C library ('conv_impl', 'use_graph', 'micro_batch'); rebuilds the device net."""
    self.net_options[name] = int(value)
    self._release()

  def _ensure_net(self, batch):
    if self._net is None or batch > self._net_batch:
      self._release()
      require_cuda()
      cap = max(batch, 1)
      self._net = self._graph.build_net(self._logits_sym, self.NUM_CLASS, self.CLASSES.index("None"), self.precision,
                                        cap, self.net_options)
      self._net_batch = cap
    return self._net

  def mc_net(self, rate, batch):
    """The stochastic net of MC dropout (``mc_dropout.forward_mc``): the same program, variables and ``net_options``
    as the default net plus one in-place dropout op per Dropout call of the model (``rate``: one float, or one per
    site).  Built on first use and cached by rate; the default net is not touched."""
    key = tuple(rate) if hasattr(rate, "__len__") else float(rate)
    handle, cap = self._mc_nets.get(key, (None, 0))
    if handle is None or batch > cap:
      if handle is not None:
        _lib.load().pcls_net_destroy(handle)
        del self._mc_nets[key]
      require_cuda()
      cap = max(batch, 1)
      handle = self._graph.build_net(self._logits_sym, self.NUM_CLASS, self.CLASSES.index("None"), self.precision, cap,
                                     self.net_options, dropout_rate=rate)
      self._mc_nets[key] = (handle, cap)
    return handle

  def forward_device(self, lidar, mask=None, mean=None, std=None, want_probabilities=True, want_logits=False,
                     out=None):
    """Runs pcls_net_forward on device tensors.  lidar: float32 CUDA tensor [B,H,W,6] (normalised, mask in channel 5)
    or, with mean/std, RAW [B,H,W,5|6] (input stage fused), or a 16-bit tensor [B,H,W,6|8] in the net's storage type
    (pcls_net_forward_in16: the normalised input already rounded, 12 / 16 bytes per pixel).  mask: uint8/bool CUDA tensor
    [B,H,W] or None.  Returns dict(predictions, probabilities?, logits?) of CUDA tensors."""
    lib = _lib.load()
    B, H, W, C = lidar.shape
    if (H, W) != (self.ZENITH_LEVEL, self.AZIMUTH_LEVEL):
      raise ValueError("input is %dx%d but the model was built for %dx%d" % (H, W, self.ZENITH_LEVEL, self.AZIMUTH_LEVEL))
    net = self._ensure_net(B)
    dev = lidar.device
    out = out or {}
    preds = out.get("predictions")
    if preds is None:
      preds = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    probs = logits = None
    if want_probabilities:
      probs = out.get("probabilities")
      if probs is None:
        probs = torch.empty((B, H, W, self.NUM_CLASS), dtype=torch.float32, device=dev)
    if want_logits:
      logits = out.get("logits")
      if logits is None:
        logits = torch.empty((B, H, W, self.NUM_CLASS), dtype=torch.float32, device=dev)
    mean_p = std_p = None
    if mean is not None:
      mean_p = (ctypes.c_double * 5)(*[float(v) for v in np.asarray(mean).reshape(-1)[:5]])
      std_p = (ctypes.c_double * 5)(*[float(v) for v in np.asarray(std).reshape(-1)[:5]])
    if mask is not None and mask.dtype == torch.bool:
      mask = mask.view(torch.uint8)
    if lidar.dtype in (torch.float16, torch.bfloat16):
      want = torch.float16 if self.precision == _lib.PCLS_F16 else torch.bfloat16
      if lidar.dtype != want or mean is not None:
        raise ValueError("a 16-bit input must be the normalised input in the net's storage type (%s)" % want)
      _lib.check(lib.pcls_net_forward_in16(net, ptr(lidar), C, ptr(mask), B, ptr(logits), ptr(probs), ptr(preds),
                                           stream_handle()), "pcls_net_forward_in16")
    else:
      _lib.check(lib.pcls_net_forward(net, ptr(lidar), C, ptr(mask), mean_p, std_p, B, ptr(logits), ptr(probs),
                                      ptr(preds), stream_handle()), "pcls_net_forward")
    res = {"predictions": preds}
    if probs is not None:
      res["probabilities"] = probs
    if logits is not None:
      res["logits"] = logits
    return res

  def input_buffers(self, batch):
    """(input8 pointer, mask pointer, frames): the device buffers a producer may write the network input into in place
    (pcls_net_input_buffers; used by the fused projection -> forward pipeline).  Builds the device net for `batch`."""
    net = self._ensure_net(batch)
    inp, msk, frames = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int()
    _lib.check(_lib.load().pcls_net_input_buffers(net, ctypes.byref(inp), ctypes.byref(msk), ctypes.byref(frames)),
               "pcls_net_input_buffers")
    return inp, msk, frames.value

  def forward_staged(self, batch, want_probabilities=True, want_logits=False, out=None):
    """Forward over an input that was written into ``input_buffers`` in place (no input kernel)."""
    H, W = self.ZENITH_LEVEL, self.AZIMUTH_LEVEL
    dev = torch.device("cuda", torch.cuda.current_device())
    out = out or {}
    preds = out.get("predictions")
    if preds is None:
      preds = torch.empty((batch, H, W), dtype=torch.int32, device=dev)
    probs = logits = None
    if want_probabilities:
      probs = out.get("probabilities")
      if probs is None:
        probs = torch.empty((batch, H, W, self.NUM_CLASS), dtype=torch.float32, device=dev)
    if want_logits:
      logits = out.get("logits")
      if logits is None:
        logits = torch.empty((batch, H, W, self.NUM_CLASS), dtype=torch.float32, device=dev)
    _lib.check(_lib.load().pcls_net_forward(self._ensure_net(batch), None, 0, None, None, None, batch, ptr(logits), ptr(probs),
                                            ptr(preds), stream_handle()), "pcls_net_forward(staged)")
    res = {"predictions": preds}
    if probs is not None:
      res["probabilities"] = probs
    if logits is not None:
      res["logits"] = logits
    return res

  def __call__(self, inputs, training=False, mask=None):
    """``probabilities, predictions = model([lidar, mask])`` (inference.py:75, eval.py:47).
    lidar [B,H,W,6] (numpy or torch, any float dtype), mask [B,H,W] bool.  Returns CUDA tensors whose ``.numpy()``
    copies to the host."""
    if training:
      raise NotImplementedError("training is outside the scope of this inference path")
    lidar_input, lidar_mask = inputs[0], inputs[1]
    # a float16 / bfloat16 lidar_input ([B,H,W,6], or [B,H,W,8] = tensor 0's layout) is shipped as it is: 12 / 16 bytes
    # per pixel over the host link instead of 24, same results as the float32 input it was rounded from
    in16 = str(getattr(lidar_input, "dtype", "")).replace("torch.", "") in ("float16", "bfloat16")
    lidar = to_device(lidar_input, lidar_input.dtype if in16 and torch.is_tensor(lidar_input) else
                      torch.float16 if in16 else torch.float32, self._pinned, "lidar")
    m = None
    if lidar_mask is not None:
      m = to_device(lidar_mask, torch.uint8 if not (torch.is_tensor(lidar_mask) and lidar_mask.dtype == torch.bool)
                    else torch.bool, self._pinned, "mask")
      m = m.reshape(lidar.shape[0], lidar.shape[1], lidar.shape[2])  # tf.squeeze(lidar_mask) semantics
    res = self.forward_device(lidar, m)
    ready = torch.cuda.Event()
    ready.record(torch.cuda.current_stream())
    return wrap(res["probabilities"], ready), wrap(res["predictions"], ready)

  def predict_raw(self, samples):
    """The per-sample body of inference.py (:47-78) for a batch, in one call: ``samples`` [B,H,W,5|6] RAW range images
    (x, y, z, intensity, depth[, label]) as the converters store them (numpy float32 / float64 or a CUDA tensor) ->
    ``(probabilities, predictions)``.  The mask / normalise / zero-fill stage runs on the device inside the forward, so
    the host ships 20 bytes per pixel (5 float32 channels) instead of the 25 of the normalised [B,H,W,6] input + mask."""
    from ..device import samples_to_device
    x = samples_to_device(samples, self._pinned, "raw")
    res = self.forward_device(x, None, mean=self.mc.INPUT_MEAN, std=self.mc.INPUT_STD)
    ready = torch.cuda.Event()
    ready.record(torch.cuda.current_stream())
    return wrap(res["probabilities"], ready), wrap(res["predictions"], ready)

  def predict_step(self, data):
    (lidar_input, lidar_mask), _, _ = data
    return self([lidar_input, lidar_mask], training=False)

  # ---- validation side, forward only (nets/SegmentationNetwork.py:71-91, :49, :118-131): one kernel
  # (csrc/validation.cu, pcls_validation_update) reads the forward's outputs once and accumulates the loss sums and the
  # class-weighted confusion matrix in float64 ----
  def _validation_update(self, loss_kind, probabilities, label, lidar_mask=None, weight=None, predictions=None, cm=None,
                         dropped=None):
    """-> float64 CUDA tensor [2] = (loss numerator, loss denominator) of this call."""
    nc = self.NUM_CLASS
    probs = _dev(probabilities, torch.float32).reshape(-1, nc).contiguous()
    y = _dev(label, torch.int32).reshape(-1).contiguous()
    n = y.numel()
    if probs.shape[0] != n:
      raise ValueError("label and probabilities sizes differ: %d vs %d" % (n, probs.shape[0]))
    m = None if lidar_mask is None else _dev(lidar_mask, torch.uint8).reshape(-1).contiguous()
    w = None if weight is None else _dev(weight, torch.float32).reshape(-1).contiguous()
    q = None if predictions is None else _dev(predictions, torch.int32).reshape(-1).contiguous()
    for name, t in (("mask", m), ("weight", w), ("predictions", q)):
      if t is not None and t.numel() != n:
        raise ValueError("%s and label sizes differ: %d vs %d" % (name, t.numel(), n))
    acc = torch.zeros(2, dtype=torch.float64, device=y.device)
    _lib.check(_lib.load().pcls_validation_update(ptr(probs), ptr(y), ptr(q), ptr(m), ptr(w), n, nc, loss_kind,
                                                  float(self.mc.DENOM_EPSILON), float(self.mc.FOCAL_GAMMA), ptr(acc),
                                                  ptr(cm), ptr(dropped), stream_handle()), "pcls_validation_update")
    return acc

  def focal_loss(self, probabilities, lidar_mask, label, loss_weight):
    """sum((1 - p)^gamma * onehot * -log(p) * w * mask) / sum(mask) * CLS_LOSS_COEF with p = probabilities +
    DENOM_EPSILON (nets/SegmentationNetwork.py:71-91)."""
    acc = self._validation_update(1, probabilities, label, lidar_mask, loss_weight)
    return acc[0] / acc[1] * float(self.mc.CLS_LOSS_COEF)

  def scc_loss(self, label, probabilities, weight):
    """tf.keras.losses.SparseCategoricalCrossentropy() on probabilities with sample weights (:49, :125): Keras clips
    the probabilities to [1e-7, 1 - 1e-7], takes -log_softmax(log p)[label] (i.e. renormalises the clipped row),
    multiplies by the weight and averages over ALL elements (SUM_OVER_BATCH_SIZE)."""
    acc = self._validation_update(2, probabilities, label, None, weight)
    return acc[0] / acc[1]

  def test_step(self, data):
    """Forward, loss and weighted MeanIoU update (nets/SegmentationNetwork.py:118-131): the forward, then ONE kernel
    over its outputs for the loss sums and the weighted confusion matrix."""
    (lidar_input, lidar_mask), label, weight = data
    probabilities, predictions = self([lidar_input, lidar_mask], training=False)
    focal = bool(self.mc.USE_FOCAL_LOSS)
    tracker = self.miou_tracker
    acc = self._validation_update(1 if focal else 2, probabilities, label, lidar_mask if focal else None, weight,
                                  predictions, tracker.weighted_cm(), tracker._dropped)
    loss = acc[0] / acc[1] * (float(self.mc.CLS_LOSS_COEF) if focal else 1.0)
    self._loss_sum += float(loss)
    self._loss_count += 1
    return {'loss': np.float32(self._loss_sum / self._loss_count), 'miou': tracker.result()}

  @property
  def metrics(self):
    return [self.miou_tracker]

  def get_config(self):
    return {"mc": self.mc}

  @classmethod
  def from_config(cls, config):
    return cls(**config)
