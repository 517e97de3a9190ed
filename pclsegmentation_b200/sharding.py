"""Frame sharding across the GPUs of one box + the single collective of the path.

Every frame / scan is independent (the reference loops one sample at a time: inference.py:44, eval.py:45,
dataset_convert/semantic_kitti.py:152), so ranks take contiguous slices of the frame list and never talk - except
for eval's confusion matrix, which is summed once with ncclAllReduce(int64) (pcls_confusion_allreduce).
One process per GPU (torchrun); ``torch.distributed`` is used only to hand the NCCL unique id around.
"""
import ctypes
import os

import torch
import torch.distributed as dist

from . import _lib
from .device import ptr, stream_handle


def shard_range(n_items, rank, world_size):
  """Contiguous, balanced slice [lo, hi) of ``n_items`` for ``rank`` (first ``n % world`` ranks get one extra)."""
  if world_size < 1 or not (0 <= rank < world_size):
    raise ValueError("bad rank/world_size %r/%r" % (rank, world_size))
  base, extra = divmod(int(n_items), world_size)
  lo = rank * base + min(rank, extra)
  return lo, lo + base + (1 if rank < extra else 0)


def env_rank():
  return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class Communicator:
  """All-reduce of the int64 confusion matrix.

  CUDA tensors: our own NCCL communicator (created through the C ABI, unique id broadcast over the default
  ``torch.distributed`` group) and ``pcls_confusion_allreduce`` on the current stream.
  CPU tensors (host-side logic under test with the gloo backend): ``torch.distributed.all_reduce``.
  """

  def __init__(self):
    self.rank = dist.get_rank() if dist.is_initialized() else 0
    self.world_size = dist.get_world_size() if dist.is_initialized() else 1
    self._comm = None

  def _ensure_nccl(self):
    if self._comm is not None or self.world_size == 1:
      return
    lib = _lib.load()
    uid = ctypes.create_string_buffer(_lib.NCCL_UNIQUE_ID_BYTES)
    if self.rank == 0:
      _lib.check(lib.pcls_comm_unique_id(uid), "pcls_comm_unique_id")
    holder = [uid.raw]
    dist.broadcast_object_list(holder, src=0)
    comm = ctypes.c_void_p()
    _lib.check(lib.pcls_comm_init(ctypes.byref(comm), self.world_size, holder[0], self.rank), "pcls_comm_init")
    self._comm = comm

  def allreduce_confusion(self, cm):
    """In-place sum of the [NC,NC] int64 matrix over all ranks."""
    if cm.dtype != torch.int64 or cm.dim() != 2 or cm.shape[0] != cm.shape[1]:
      raise TypeError("confusion matrix must be a square int64 tensor")
    if self.world_size == 1:
      return cm
    if cm.is_cuda:
      self._ensure_nccl()
      _lib.check(_lib.load().pcls_confusion_allreduce(ptr(cm), cm.shape[0], self._comm, stream_handle()),
                 "pcls_confusion_allreduce")
    else:
      dist.all_reduce(cm, op=dist.ReduceOp.SUM)
    return cm

  def allreduce_aux(self, metric):
    """The parts of a MeanIoU that are not the int64 matrix: ``_cmw`` (float64, weighted updates) and ``_dropped``.
    Ranks agree first on whether anyone holds a weighted matrix (a rank that never saw a weighted update has none)."""
    if self.world_size == 1:
      return
    dev = metric._cm.device
    has_w = torch.tensor([1 if metric._cmw is not None else 0], dtype=torch.int64, device=dev)
    dist.all_reduce(has_w, op=dist.ReduceOp.MAX)
    if int(has_w.item()):
      if metric._cmw is None:
        metric._cmw = torch.zeros(tuple(metric._cm.shape), dtype=torch.float64, device=dev)
      dist.all_reduce(metric._cmw, op=dist.ReduceOp.SUM)
    dist.all_reduce(metric._dropped, op=dist.ReduceOp.SUM)

  def allreduce_sums(self, tensors):
    """In-place sum of each tensor over all ranks with ``torch.distributed`` (small accumulators, off the hot path)."""
    if self.world_size == 1:
      return
    for t in tensors:
      dist.all_reduce(t, op=dist.ReduceOp.SUM)

  def close(self):
    if self._comm is not None:
      _lib.load().pcls_comm_destroy(self._comm)
      self._comm = None
