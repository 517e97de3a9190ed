"""Symbolic layer toolkit for the model builders.

The reference's ``nets/*.py`` are Keras models: ``call`` chains ``tf.keras.layers`` objects and Keras traces that
into a graph.  Here ``call`` chains the small stand-ins below over *symbolic* tensors; the trace is an op program in
which ``conv -> BatchNormalization -> activation -> (+ residual) -> concat`` chains are folded into ONE fused
convolution op of libpclseg (BN folded into the weights, activation / residual adds in the epilogue, ``tf.concat`` as
a channel-offset write).  ``build_net`` then hands the program and the Keras-named variables to the C ABI
(pcls_net_tensor / pcls_net_conv / pcls_net_maxpool3x3_s2 / pcls_net_cam).

Variables are keyed by their Keras attribute path (SURVEY.md Appendix C), e.g. ``fire2/squeeze/kernel``.
"""
import ctypes

import numpy as np

from .. import _lib

BN_EPS = 1e-3  # tf.keras.layers.BatchNormalization default; the reference never passes epsilon=


class Sym:
  """Symbolic NHWC activation ``[B, H, width, channels]``."""

  def __init__(self, graph, width, channels, producers=(), logits=False, is_input=False):
    self.graph, self.width, self.channels = graph, width, channels
    self.producers = list(producers)  # pending fused-conv ops that write this tensor
    self.logits = logits
    self.is_input = is_input
    self.consumed = False
    self.tid = None

  # run_enc_block / run_dec_block look at y.shape[1] / y.shape[2] (nets/Darknet.py:263-277)
  @property
  def shape(self):
    return (None, self.graph.H, self.width, self.channels)

  def __add__(self, other):
    return self.graph.add(self, other)

  __iadd__ = __add__


class Graph:
  def __init__(self, H, W):
    self.H, self.W = H, W
    self.variables = {}     # name -> np.float32 array (Keras layout)
    self.program = []       # ops in execution order
    self.dropout_sites = []  # (sym, rate, op it follows) per Dropout call, in trace order (MC dropout sites)
    self.rng = np.random.default_rng(0)
    self.merge_expand = True  # fuse Fire expand1x1 || expand3x3 into one convolution (see concat)
    self.input = Sym(self, W, 8, is_input=True)

  # ---- variables ---------------------------------------------------------------------------------
  def variable(self, name, shape, init):
    if name not in self.variables:
      if init == "glorot":
        receptive = int(np.prod(shape[:-2]))
        fan_in, fan_out = shape[-2] * receptive, shape[-1] * receptive
        limit = np.sqrt(6.0 / (fan_in + fan_out))
        val = self.rng.uniform(-limit, limit, size=shape)
      elif init == "ones":
        val = np.ones(shape)
      else:
        val = np.zeros(shape)
      self.variables[name] = val.astype(np.float32)
    return name

  # ---- ops ---------------------------------------------------------------------------------------
  def _consume(self, x):
    x.consumed = True
    return x

  def conv(self, x, name, kind, kh, kw, stride_w, cout, use_bias):
    self._consume(x)
    cin = 6 if x.is_input else x.channels  # the mask is input channel 5; channels 6,7 are zero padding
    if kind == _lib.KIND_CONV:
      kshape, wout = (kh, kw, cin, cout), (x.width + stride_w - 1) // stride_w
    else:
      kshape, wout = (kh, kw, cout, cin), x.width * 2
    op = dict(op="conv", kind=kind, kh=kh, kw=kw, stride_w=stride_w, cin=cin, cout=cout,
              kernel=self.variable(name + "/kernel", kshape, "glorot"),
              bias=self.variable(name + "/bias", (cout,), "zeros") if use_bias else None,
              bn=None, act=_lib.ACT_NONE, src=x, dst=None, off=0, res=[], stage=0)
    self.program.append(op)
    out = Sym(self, wout, cout, producers=[op])
    op["dst"] = out
    return out

  def batch_norm(self, x, name):
    assert len(x.producers) == 1 and x.producers[0]["stage"] == 0 and not x.consumed, \
        "BatchNormalization must directly follow a convolution"
    op = x.producers[0]
    c = op["cout"]
    for v, init in (("gamma", "ones"), ("beta", "zeros"), ("moving_mean", "zeros"), ("moving_variance", "ones")):
      self.variable(name + "/" + v, (c,), init)
    op["bn"], op["stage"] = name, 1
    return x

  def activation(self, x, act):
    assert x.producers and not x.consumed and all(p["stage"] <= 1 for p in x.producers), \
        "activation must follow conv(+BN) directly"
    for p in x.producers:
      p["act"], p["stage"] = act, 2
    return x

  def add(self, a, b):
    """x += residual / tf.add(x, skip): folded into the epilogue of the conv(s) producing ``a``."""
    if not a.producers or a.consumed:
      a, b = b, a
    assert a.producers and not a.consumed, "add: one operand must be an unconsumed convolution output"
    assert b.width == a.width and b.channels == a.channels and not b.logits
    self._consume(b)
    for p in a.producers:
      assert len(p["res"]) < 2, "at most two residual adds per convolution"
      p["res"].append(b)
      p["stage"] = 3
    return a

  def concat(self, parts):
    """tf.concat(axis=3) of fresh convolution outputs: they write channel slices of one tensor.

    Fire expand pairs (expand1x1 || expand3x3 on the same squeeze output, nets/SqueezeSegV2.py:124-127, 196-199) are
    MERGED into one 3x3 convolution with N = E1 + E3 output channels whose first E1 channels carry the 1x1 weights in
    the centre tap: the squeeze tensor is read once, every output pixel row (and every residual row) is touched by ONE
    kernel as a full contiguous line instead of two half lines, and a launch disappears.  Done when N <= 256."""
    assert all(len(p.producers) == 1 and not p.consumed for p in parts)
    out = Sym(self, parts[0].width, sum(p.channels for p in parts))
    ops = [p.producers[0] for p in parts]
    if (self.merge_expand and len(ops) == 2 and all(o["op"] == "conv" and o["kind"] == _lib.KIND_CONV for o in ops) and
        ops[0]["src"] is ops[1]["src"] and (ops[0]["kh"], ops[0]["kw"]) == (1, 1) and (ops[1]["kh"], ops[1]["kw"]) == (3, 3) and
        ops[0]["stride_w"] == 1 and ops[1]["stride_w"] == 1 and ops[0]["act"] == ops[1]["act"] and
        (ops[0]["bn"] is None) == (ops[1]["bn"] is None) and (ops[0]["bias"] is None) == (ops[1]["bias"] is None) and
        not ops[0]["res"] and not ops[1]["res"] and out.channels <= 256):
      a, b = ops
      merged = dict(op="conv", kind=_lib.KIND_CONV, kh=3, kw=3, stride_w=1, cin=a["cin"], cout=out.channels,
                    kernel=None, bias=None, bn=None, merge=(a, b), act=a["act"], src=a["src"], dst=out, off=0, res=[],
                    stage=max(a["stage"], b["stage"]))
      i = self.program.index(a)
      self.program.remove(b)
      self.program[i] = merged
      out.producers.append(merged)
      return out
    off = 0
    for p in parts:
      assert p.width == out.width
      op = p.producers[0]
      op["dst"], op["off"] = out, off
      out.producers.append(op)
      off += p.channels
    return out

  def _merged_arrays(self, op):
    """(kernel [3,3,Cin,E1+E3], bias, gamma, beta, mean, var) of a merged Fire expand pair, from the current variables."""
    a, b = op["merge"]
    v = self.variables
    k1, k3 = v[a["kernel"]], v[b["kernel"]]
    kernel = np.zeros((3, 3, k3.shape[2], k1.shape[3] + k3.shape[3]), np.float32)
    kernel[1, 1, :, :k1.shape[3]] = k1[0, 0]
    kernel[:, :, :, k1.shape[3]:] = k3
    cat = lambda x, y: np.concatenate([v[x], v[y]]).astype(np.float32)
    bias = cat(a["bias"], b["bias"]) if a["bias"] else None
    bn = [cat(a["bn"] + s, b["bn"] + s) for s in ("/gamma", "/beta", "/moving_mean", "/moving_variance")] if a["bn"] else [None] * 4
    return [kernel, bias] + bn

  def dropout(self, x, rate):
    """Records a Dropout call as an MC dropout site and returns ``x``: the traced program does not change.  A net built
    with a ``dropout_rate`` drops ``x`` in place right after the last op traced so far (the op object is recorded, not
    its index, so that a later merge of program entries cannot move the site), and every later reader sees the dropped
    tensor; nothing may be folded into its producer after this point."""
    assert self.program and not x.is_input, "a dropout site must follow the op that writes its tensor"
    self._consume(x)
    self.dropout_sites.append((x, float(rate), self.program[-1]))
    return x

  def max_pool_3x3_s2(self, x):
    self._consume(x)
    out = Sym(self, (x.width + 1) // 2, x.channels)
    self.program.append(dict(op="pool", src=x, dst=out))
    return out

  def cam(self, x, name, reduced):
    self._consume(x)
    c = x.channels
    for sub, shape in (("squeeze", (1, 1, c, reduced)), ("excitation", (1, 1, reduced, c))):
      self.variable(f"{name}/{sub}/kernel", shape, "glorot")
      self.variable(f"{name}/{sub}/bias", (shape[-1],), "zeros")
      for v, init in (("gamma", "ones"), ("beta", "zeros"), ("moving_mean", "zeros"), ("moving_variance", "ones")):
        self.variable(f"{name}/{sub}_bn/{v}", (shape[-1],), init)
    out = Sym(self, x.width, c)
    self.program.append(dict(op="cam", name=name, channels=c, reduced=reduced, src=x, dst=out))
    return out

  # ---- lowering to the C ABI -----------------------------------------------------------------------
  def build_net(self, logits, num_classes, none_index, precision, max_batch, options=None, dropout_rate=None):
    """Emits the traced program into a fresh pcls_net and finalizes it.  Returns the handle (c_void_p).
    ``dropout_rate``: None (the deterministic net), one rate for every site of ``dropout_sites``, or a sequence with one
    rate per site; each site becomes a pcls_net_dropout op (site = its index) right after the op it follows."""
    rates = None
    if dropout_rate is not None:
      rates = [float(r) for r in dropout_rate] if hasattr(dropout_rate, "__len__") else \
          [float(dropout_rate)] * len(self.dropout_sites)
      if len(rates) != len(self.dropout_sites):
        raise ValueError("%d dropout rates for %d sites" % (len(rates), len(self.dropout_sites)))
      lost = [k for k, (_, _, after) in enumerate(self.dropout_sites) if not any(op is after for op in self.program)]
      if lost:
        raise ValueError("dropout sites %s follow ops that are no longer in the program" % lost)
    lib = _lib.load()
    handle = ctypes.c_void_p()
    _lib.check(lib.pcls_net_create(ctypes.byref(handle), self.H, self.W, precision, max_batch), "pcls_net_create")
    try:
      for k, v in (options or {}).items():
        _lib.check(lib.pcls_net_set_option(handle, k.encode(), int(v)), "pcls_net_set_option(%s)" % k)
      self.input.tid = 0
      keep = []  # keep ctypes-owned host arrays alive until finalize

      def fptr(name):
        if name is None:
          return None
        a = np.ascontiguousarray(self.variables[name], dtype=np.float32)
        keep.append(a)
        return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))

      def aptr(a):
        if a is None:
          return None
        a = np.ascontiguousarray(a, dtype=np.float32)
        keep.append(a)
        return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))

      def tid(sym):
        if sym.tid is None:
          sym.tid = _lib.check(lib.pcls_net_tensor(handle, sym.width, sym.channels, 1 if sym.logits else 0),
                               "pcls_net_tensor")
        return sym.tid

      for s in self._all_syms():
        s.tid = None
      self.input.tid = 0
      logits.logits = True

      def emit_dropouts(prev):
        for k, (sym, _, after) in enumerate(self.dropout_sites):
          if rates is not None and after is prev:
            _lib.check(lib.pcls_net_dropout(handle, tid(sym), k, rates[k]), "pcls_net_dropout(site %d)" % k)

      for i, op in enumerate(self.program):
        emit_dropouts(self.program[i - 1] if i else None)
        if op["op"] == "conv":
          d = _lib.ConvDesc()
          d.kind, d.kh, d.kw, d.stride_w, d.cin, d.cout = op["kind"], op["kh"], op["kw"], op["stride_w"], op["cin"], op["cout"]
          if op.get("merge"):
            arrs = [aptr(x) for x in self._merged_arrays(op)]
            d.h_kernel, d.h_bias, d.h_bn_gamma, d.h_bn_beta, d.h_bn_mean, d.h_bn_var = arrs
          else:
            d.h_kernel, d.h_bias = fptr(op["kernel"]), fptr(op["bias"])
            bn = op["bn"]
            d.h_bn_gamma = fptr(bn + "/gamma" if bn else None)
            d.h_bn_beta = fptr(bn + "/beta" if bn else None)
            d.h_bn_mean = fptr(bn + "/moving_mean" if bn else None)
            d.h_bn_var = fptr(bn + "/moving_variance" if bn else None)
          d.bn_eps, d.act = BN_EPS, op["act"]
          d.in_tensor, d.out_tensor, d.out_channel_offset = tid(op["src"]), tid(op["dst"]), op["off"]
          res = [tid(r) for r in op["res"]] + [-1, -1]
          d.residual0, d.residual1 = res[0], res[1]
          d.out_is_logits = 1 if op["dst"].logits else 0
          _lib.check(lib.pcls_net_conv(handle, ctypes.byref(d)), "pcls_net_conv(%s)" % (op["kernel"] or op["merge"][1]["kernel"]))
        elif op["op"] == "pool":
          _lib.check(lib.pcls_net_maxpool3x3_s2(handle, tid(op["src"]), tid(op["dst"])), "pcls_net_maxpool3x3_s2")
        else:
          d = _lib.CamDesc()
          n = op["name"]
          d.channels, d.reduced, d.bn_eps = op["channels"], op["reduced"], BN_EPS
          d.h_sq_kernel, d.h_sq_bias = fptr(n + "/squeeze/kernel"), fptr(n + "/squeeze/bias")
          d.h_sq_gamma, d.h_sq_beta = fptr(n + "/squeeze_bn/gamma"), fptr(n + "/squeeze_bn/beta")
          d.h_sq_mean, d.h_sq_var = fptr(n + "/squeeze_bn/moving_mean"), fptr(n + "/squeeze_bn/moving_variance")
          d.h_ex_kernel, d.h_ex_bias = fptr(n + "/excitation/kernel"), fptr(n + "/excitation/bias")
          d.h_ex_gamma, d.h_ex_beta = fptr(n + "/excitation_bn/gamma"), fptr(n + "/excitation_bn/beta")
          d.h_ex_mean, d.h_ex_var = fptr(n + "/excitation_bn/moving_mean"), fptr(n + "/excitation_bn/moving_variance")
          d.in_tensor, d.out_tensor = tid(op["src"]), tid(op["dst"])
          _lib.check(lib.pcls_net_cam(handle, ctypes.byref(d)), "pcls_net_cam(%s)" % n)
      emit_dropouts(self.program[-1])
      _lib.check(lib.pcls_net_finalize(handle, tid(logits), num_classes, none_index), "pcls_net_finalize")
    except Exception:
      lib.pcls_net_destroy(handle)
      raise
    return handle

  def _all_syms(self):
    seen = []
    for op in self.program:
      for s in [op["src"], op["dst"]] + list(op.get("res", [])):
        if s not in seen:
          seen.append(s)
    return seen


# ---- Keras-like layer objects ------------------------------------------------------------------------
class Layer:
  """Base of the stand-ins; ``path`` is the Keras attribute path of the layer inside the model."""

  def __init__(self, path):
    self.path = path


class Conv2D(Layer):
  """tf.keras.layers.Conv2D(filters, kernel_size, strides=[1,s], padding='SAME'|'VALID' for 1x1, use_bias)."""

  def __init__(self, path, filters, kernel_size, strides=1, use_bias=True):
    super().__init__(path)
    self.filters, self.use_bias = filters, use_bias
    self.kernel_size = (kernel_size, kernel_size) if isinstance(kernel_size, int) else tuple(kernel_size)
    self.strides = (strides, strides) if isinstance(strides, int) else tuple(strides)
    assert self.strides[0] == 1, "the reference never strides along H"

  def __call__(self, x):
    return x.graph.conv(x, self.path, _lib.KIND_CONV, self.kernel_size[0], self.kernel_size[1], self.strides[1],
                        self.filters, self.use_bias)


class Conv2DTranspose(Layer):
  """tf.keras.layers.Conv2DTranspose(filters, kernel_size=[1,4], strides=[1,2], padding='SAME')."""

  def __init__(self, path, filters, kernel_size=(1, 4), strides=(1, 2), use_bias=True):
    super().__init__(path)
    assert tuple(kernel_size) == (1, 4) and tuple(strides) == (1, 2)
    self.filters, self.use_bias = filters, use_bias

  def __call__(self, x):
    return x.graph.conv(x, self.path, _lib.KIND_DECONV_1x4_S2, 1, 4, 2, self.filters, self.use_bias)


class BatchNormalization(Layer):
  def __call__(self, x, training=False):
    return x.graph.batch_norm(x, self.path)


class LeakyReLU(Layer):
  def __init__(self, alpha=0.1):
    super().__init__(None)
    assert abs(alpha - 0.1) < 1e-12, "the kernels implement LeakyReLU(0.1), the only slope the reference uses"

  def __call__(self, x):
    return x.graph.activation(x, _lib.ACT_LEAKY)


class Dropout(Layer):
  """Identity in the default net (training=False everywhere on this path).  Each call records an MC dropout site
  (``Graph.dropout`` / ``Graph.dropout_sites``), used only by the stochastic net of ``mc_dropout``."""

  def __init__(self, rate):
    super().__init__(None)
    self.rate = rate

  def __call__(self, x, training=False):
    return x.graph.dropout(x, self.rate)


def relu(x):
  return x.graph.activation(x, _lib.ACT_RELU)


def concat(parts, axis=3):
  assert axis == 3
  return parts[0].graph.concat(parts)


def add(a, b):
  return a.graph.add(a, b)


def max_pool2d(x, ksize=3, strides=(1, 2), padding='SAME'):
  assert ksize == 3 and list(strides) == [1, 2] and padding == 'SAME'
  return x.graph.max_pool_3x3_s2(x)
