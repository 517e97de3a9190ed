"""ctypes binding of libpclseg.so (include/pclseg.h).  There is no fallback: if the library is missing or a
call fails, this module raises."""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_uint32, \
    c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpclseg%s.so" % os.environ.get("PCLS_LIB_SUFFIX", ""))  # suffix: development builds

PCLS_F16, PCLS_BF16 = 0, 1
ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
KIND_CONV, KIND_DECONV_1x4_S2 = 0, 1
NCCL_UNIQUE_ID_BYTES = 128
ABI_VERSION = 2   # include/pclseg.h PCLS_ABI_VERSION

_fp = POINTER(c_float)


class ConvDesc(Structure):
  _fields_ = [("kind", c_int), ("kh", c_int), ("kw", c_int), ("stride_w", c_int), ("cin", c_int), ("cout", c_int),
              ("h_kernel", _fp), ("h_bias", _fp), ("h_bn_gamma", _fp), ("h_bn_beta", _fp), ("h_bn_mean", _fp),
              ("h_bn_var", _fp), ("bn_eps", c_float), ("act", c_int), ("in_tensor", c_int), ("out_tensor", c_int),
              ("out_channel_offset", c_int), ("residual0", c_int), ("residual1", c_int), ("out_is_logits", c_int)]


class CamDesc(Structure):
  _fields_ = [("channels", c_int), ("reduced", c_int)] + \
             [(n, _fp) for n in ("h_sq_kernel", "h_sq_bias", "h_sq_gamma", "h_sq_beta", "h_sq_mean", "h_sq_var",
                                 "h_ex_kernel", "h_ex_bias", "h_ex_gamma", "h_ex_beta", "h_ex_mean", "h_ex_var")] + \
             [("bn_eps", c_float), ("in_tensor", c_int), ("out_tensor", c_int)]


# name -> (restype, argtypes); must list every symbol include/pclseg.h declares
SIGNATURES = {
  "pcls_abi_version": (c_int, []),
  "pcls_last_error": (c_char_p, []),
  "pcls_project_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_double, c_double,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_project_resolve": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                   c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_project_resolve_net_input": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, POINTER(c_double),
                                             POINTER(c_double), c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_point_labels": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                                c_int, c_int, c_int, c_int, POINTER(c_float), c_float, c_int, c_void_p, c_void_p,
                                c_void_p]),
  "pcls_point_instances_scratch_bytes": (c_int64, [c_int, c_int, c_int]),
  "pcls_point_instances": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p,
                                   c_void_p, c_int, c_uint32, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
  "pcls_tta_views": (c_int, [c_void_p, c_int, c_int, c_int, c_int, POINTER(c_double), POINTER(c_double), c_int,
                             POINTER(c_int), POINTER(c_int), POINTER(c_double), POINTER(c_double), c_int, c_void_p,
                             c_void_p, c_void_p]),
  "pcls_tta_merge": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, POINTER(c_int),
                             POINTER(c_int), c_void_p, c_void_p, c_void_p]),
  "pcls_confidence": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p,
                              c_void_p]),
  "pcls_temperature_nll": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, POINTER(c_float), c_void_p,
                                   c_void_p, c_void_p]),
  "pcls_reliability_update": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
  "pcls_point_confidence": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                                    c_int, c_void_p, c_void_p]),
  "pcls_net_dropout": (c_int, [c_void_p, c_int, c_int, c_double]),
  "pcls_net_set_dropout": (c_int, [c_void_p, c_uint64, c_uint64, c_int, c_void_p]),
  "pcls_mc_accumulate": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
  "pcls_mc_finalize": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p]),
  "pcls_semantic_map_vote": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_double, c_double, c_double,
                                     c_void_p, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
  "pcls_semantic_map_grow": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p,
                                     c_void_p]),
  "pcls_semantic_map_query": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_double, c_void_p, c_int, c_uint32,
                                      c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
  "pcls_map_labels":(c_int, [c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p]),
  "pcls_dataset_stats": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, POINTER(c_double), c_int, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_net_input_buffers": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int)]),
  "pcls_head": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p]),
  "pcls_cast_f64_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
  "pcls_unpack_xyzir": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
  "pcls_input_stage": (c_int, [c_void_p, c_int, c_int64, POINTER(c_double), POINTER(c_double), c_int, c_void_p,
                               c_void_p, c_void_p, POINTER(c_double), c_int, c_void_p, c_void_p]),
  "pcls_confusion_update": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
  "pcls_validation_update": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_double,
                                     c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_comm_unique_id": (c_int, [c_char_p]),
  "pcls_comm_init": (c_int, [POINTER(c_void_p), c_int, c_char_p, c_int]),
  "pcls_comm_destroy": (c_int, [c_void_p]),
  "pcls_confusion_allreduce": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
  "pcls_net_create": (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int]),
  "pcls_net_destroy": (None, [c_void_p]),
  "pcls_net_tensor": (c_int, [c_void_p, c_int, c_int, c_int]),
  "pcls_net_conv": (c_int, [c_void_p, POINTER(ConvDesc)]),
  "pcls_net_maxpool3x3_s2": (c_int, [c_void_p, c_int, c_int]),
  "pcls_net_cam": (c_int, [c_void_p, POINTER(CamDesc)]),
  "pcls_net_finalize": (c_int, [c_void_p, c_int, c_int, c_int]),
  "pcls_net_forward": (c_int, [c_void_p, c_void_p, c_int, c_void_p, POINTER(c_double), POINTER(c_double), c_int,
                               c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_net_forward_in16": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
  "pcls_net_read_tensor": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
  "pcls_net_num_ops": (c_int, [c_void_p]),
  "pcls_net_profile_ops": (c_int, [c_void_p, c_void_p, c_int, c_void_p, POINTER(c_double), POINTER(c_double), c_int,
                                   c_void_p, c_void_p, c_void_p, POINTER(c_float), c_void_p]),
  "pcls_net_op_info": (c_int, [c_void_p, c_int, c_char_p, POINTER(c_int), POINTER(c_int64), POINTER(c_int64)]),
  "pcls_net_launches_per_forward": (c_int, [c_void_p]),
  "pcls_net_workspace_bytes": (c_int64, [c_void_p]),
  "pcls_net_set_option": (c_int, [c_void_p, c_char_p, c_int]),
}

_lib = None


class PclsError(RuntimeError):
  pass


def load():
  """Loads libpclseg.so and declares every signature.  Raises if the library has not been built."""
  global _lib
  if _lib is not None:
    return _lib
  if not os.path.exists(LIB_PATH):
    raise PclsError("libpclseg.so is not built (%s missing): run `python -m pclsegmentation_b200.build` "
                    "or __graft_entry__.build().  There is no CPU fallback." % LIB_PATH)
  lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
  for name, (res, args) in SIGNATURES.items():
    fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
    fn.restype = res
    fn.argtypes = args
  if lib.pcls_abi_version() != ABI_VERSION:
    raise PclsError("libpclseg.so ABI version %d, expected %d" % (lib.pcls_abi_version(), ABI_VERSION))
  _lib = lib
  return lib


def check(status, what=""):
  """Turns a negative pcls_status into an exception carrying pcls_last_error()."""
  if status < 0:
    msg = load().pcls_last_error()
    raise PclsError("%s failed (%d): %s" % (what or "libpclseg call", status, (msg or b"").decode()))
  return status
