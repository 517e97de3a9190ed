"""Dataset statistics on the GPU: per-channel mean / std (the numbers behind a config's ``INPUT_MEAN`` / ``INPUT_STD``),
channel ranges, pixel occupancy per beam row and per column, and class frequencies - from converted ``[H,W,6]`` range
images or straight from raw scans.  The reference computes the mean / std offline with numpy
(``preprocessing/inspect_training_data.py``); this is the project's own contract, bit parity with its ``RunningStd`` is
not claimed.

    python -m pclsegmentation_b200.dataset_stats -d 'out/train/*.npy' -n squeezesegv2kitti [-b 64] [--json stats.json]
    python -m pclsegmentation_b200.dataset_stats --scans 'seq/0[0-7]/velodyne/*.bin' --format kitti --width 2048 \\
        [--labels '.../*.label' --learning_map semantic-kitti.yaml] -n squeezesegv2kitti
    torchrun --nproc-per-node 8 -m pclsegmentation_b200.dataset_stats ...      # files sharded over 8 GPUs

Each frame is reduced on the GPU (``pcls_dataset_stats``) to one row of float64 sums per channel - sum(d), sum(d*d),
min, max with d = x - shift, over the valid pixels (range > 0) - in an order that depends only on the frame's shape.
The frames' rows are combined on the host with ``math.fsum``, which is exact and so independent of the order: the
result is the same bits for any batch size and any number of GPUs.  The shift defaults to the config's ``INPUT_MEAN``,
which keeps d small and the variance free of cancellation.
"""
import argparse
import glob
import json
import math

import numpy as np

# finish() keys, documented for the --json file
KEYS = ("frames", "pixels", "valid", "valid_fraction", "mean", "std", "min", "max", "row_valid_fraction",
        "col_valid_fraction", "class_pixels", "class_frequency", "dropped", "shift")


def combine(state, shift, H, W):
  """Host combination of the per-frame rows ``state`` (frame_sums [F,5,4], frame_valid [F], row_valid [H],
  col_valid [W], class_pixels [NC], dropped) into the report ``DatasetStats.finish`` returns."""
  sums = np.asarray(state["frame_sums"], np.float64).reshape(-1, 5, 4)
  fv = np.asarray(state["frame_valid"], np.int64).reshape(-1)
  F = int(fv.shape[0])
  n = int(fv.sum())
  s = np.asarray(shift, np.float64).reshape(5)
  mean = np.full(5, np.nan)
  std = np.full(5, np.nan)
  if n > 0:
    for c in range(5):
      m1 = math.fsum(sums[:, c, 0].tolist()) / n
      m2 = math.fsum(sums[:, c, 1].tolist()) / n
      mean[c] = s[c] + m1
      std[c] = math.sqrt(max(m2 - m1 * m1, 0.0))          # population std
  cls = np.asarray(state["class_pixels"], np.int64)
  ncls = int(cls.sum())
  return dict(frames=F, pixels=F * H * W, valid=n, valid_fraction=n / (F * H * W) if F else float("nan"),
              mean=mean.reshape(1, 1, 5), std=std.reshape(1, 1, 5),
              min=sums[:, :, 2].min(0, initial=np.inf), max=sums[:, :, 3].max(0, initial=-np.inf),
              row_valid_fraction=np.asarray(state["row_valid"], np.int64) / max(F * W, 1),
              col_valid_fraction=np.asarray(state["col_valid"], np.int64) / max(F * H, 1),
              class_pixels=cls, class_frequency=cls / ncls if ncls else np.zeros(cls.shape),
              dropped=int(state["dropped"]), shift=s.reshape(1, 1, 5))


def gather(state, comm):
  """Every rank's per-frame rows and the sums of the integer counters, on every rank (torch.distributed; the order of
  the rows does not matter to ``combine``)."""
  if comm is None or comm.world_size == 1:
    return state
  import torch.distributed as dist
  parts = [None] * comm.world_size
  dist.all_gather_object(parts, state)
  return dict(frame_sums=np.concatenate([p["frame_sums"] for p in parts]),
              frame_valid=np.concatenate([p["frame_valid"] for p in parts]),
              row_valid=sum(p["row_valid"] for p in parts), col_valid=sum(p["col_valid"] for p in parts),
              class_pixels=sum(p["class_pixels"] for p in parts), dropped=sum(int(p["dropped"]) for p in parts))


class DatasetStats:
  """Accumulates the statistics of ``[B,H,W,5|6]`` range images batch by batch on the current CUDA device.

  ``mc_or_num_classes``: a config (``mc``: classes, ``INPUT_MEAN`` as the default shift) or a class count (shift 0).
  """

  def __init__(self, mc_or_num_classes, H, W, shift=None):
    if isinstance(mc_or_num_classes, (int, np.integer)):
      self.num_classes, default_shift = int(mc_or_num_classes), np.zeros(5)
    else:
      self.num_classes, default_shift = int(mc_or_num_classes.NUM_CLASS), mc_or_num_classes.INPUT_MEAN
    if not 1 <= self.num_classes <= 32:
      raise ValueError("num_classes %d not in [1, 32]" % self.num_classes)
    self.H, self.W = int(H), int(W)
    self.shift = np.ascontiguousarray(np.asarray(default_shift if shift is None else shift, np.float64).reshape(5))
    self._sums, self._valid = [], []
    self._counts = None
    self._pinned = {}                       # host staging buffer of update()

  def _run(self, frames, count_labels):
    import ctypes
    import torch
    from . import _lib
    from .device import ptr, stream_handle
    B, H, W, C = frames.shape
    dev = frames.device
    if self._counts is None:
      self._counts = {k: torch.zeros(n, dtype=torch.int64, device=dev)
                      for k, n in (("row_valid", self.H), ("col_valid", self.W), ("class_pixels", self.num_classes),
                                   ("dropped", 1))}
    sums = torch.empty((B, 5, 4), dtype=torch.float64, device=dev)
    valid = torch.empty(B, dtype=torch.int64, device=dev)
    k = self._counts
    _lib.check(_lib.load().pcls_dataset_stats(
        ptr(frames), 1 if frames.dtype == torch.float64 else 0, C, B, H, W,
        self.shift.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), self.num_classes, ptr(sums), ptr(valid),
        ptr(k["row_valid"]), ptr(k["col_valid"]), ptr(k["class_pixels"]) if count_labels else None,
        ptr(k["dropped"]) if count_labels else None, stream_handle()), "pcls_dataset_stats")
    self._sums.append(sums)
    self._valid.append(valid)
    return sums, valid

  def update(self, frames, count_labels=True):
    """frames: ``[B,H,W,5|6]`` numpy float32 / float64 or a torch tensor of either (CPU or CUDA).  float64 stays float64
    on the device.  6-channel frames also count their label channel unless ``count_labels`` is False (files converted
    without label files carry 0 there, which would count every valid pixel as class 0).  Returns the batch's device rows
    (frame_sums [B,5,4] float64, frame_valid [B] int64)."""
    import torch
    from .device import to_device
    if torch.is_tensor(frames):
      dt = frames.dtype
    else:
      frames = np.asarray(frames)
      dt = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}.get(frames.dtype)
    if dt not in (torch.float32, torch.float64):
      raise TypeError("frames must be float32 or float64, got %s" % frames.dtype)
    if len(frames.shape) != 4 or tuple(frames.shape[1:3]) != (self.H, self.W) or frames.shape[3] not in (5, 6):
      raise ValueError("frames must be [B,%d,%d,5|6], got %s" % (self.H, self.W, tuple(frames.shape)))
    d = to_device(frames, dt, self._pinned, "frames")
    return self._run(d, count_labels and d.shape[3] == 6)

  def update_scans(self, batch, projector, use_ring=False):
    """batch: the dict ``dataset_convert.ScanBatchLoader.load`` returns.  The scans are projected on the device with the
    converters' settings (``empty_fill=0``, labels through the projector's learning map) and the float32 images are
    reduced like ``.npy`` files - nothing is written.  Labels are counted only when the batch has label files."""
    if (projector.H, projector.W) != (self.H, self.W):
      raise ValueError("projector is %dx%d, statistics are %dx%d" % (projector.H, projector.W, self.H, self.W))
    out = projector.project(batch["points"], batch["offsets"], labels=batch["labels"],
                            ring=batch["ring"] if use_ring else None, empty_fill=0.0, want_idx=False)
    return self._run(out["image"], batch["labels"] is not None)

  def state(self):
    """This rank's per-frame rows and integer counters as numpy arrays."""
    import torch
    if not self._sums:
      return dict(frame_sums=np.zeros((0, 5, 4)), frame_valid=np.zeros(0, np.int64), row_valid=np.zeros(self.H, np.int64),
                  col_valid=np.zeros(self.W, np.int64), class_pixels=np.zeros(self.num_classes, np.int64), dropped=0)
    k = self._counts
    return dict(frame_sums=torch.cat(self._sums).cpu().numpy(), frame_valid=torch.cat(self._valid).cpu().numpy(),
                row_valid=k["row_valid"].cpu().numpy(), col_valid=k["col_valid"].cpu().numpy(),
                class_pixels=k["class_pixels"].cpu().numpy(), dropped=int(k["dropped"].item()))

  def finish(self, comm=None):
    """The statistics over every frame seen (on every rank with ``comm``, a ``sharding.Communicator``): frames, pixels,
    valid; mean / std float64 [1,1,5] like ``mc.INPUT_MEAN`` (population std); per-channel min / max; row / column
    valid fractions; class_pixels, class_frequency (class_pixels over their sum: the dropped pixels are not in it),
    dropped (valid pixels whose label is not a class id)."""
    return combine(gather(self.state(), comm), self.shift, self.H, self.W)


def to_json(rep):
  return {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in rep.items()}


def config_check(rep, mc):
  """(mean - mc.INPUT_MEAN) / mc.INPUT_STD and std / mc.INPUT_STD per channel: about 0 and 1 on data that matches."""
  ref_m = np.asarray(mc.INPUT_MEAN, np.float64).reshape(5)
  ref_s = np.asarray(mc.INPUT_STD, np.float64).reshape(5)
  return (rep["mean"].reshape(5) - ref_m) / ref_s, rep["std"].reshape(5) / ref_s


def print_report(rep, mc, config_name):
  np.set_printoptions(linewidth=200)
  chans = ("x", "y", "z", "remission", "range")
  fmt = lambda a: ", ".join(repr(float(x)) for x in np.asarray(a).reshape(-1))
  print("%d frames, %d of %d pixels valid (%.4f)" % (rep["frames"], rep["valid"], rep["pixels"], rep["valid_fraction"]))
  print("mc.INPUT_MEAN = np.array([[[%s]]])" % fmt(rep["mean"]))
  print("mc.INPUT_STD = np.array([[[%s]]])" % fmt(rep["std"]))
  print("%-10s %14s %14s" % ("channel", "min", "max"))
  for c, name in enumerate(chans):
    print("%-10s %14.6g %14.6g" % (name, rep["min"][c], rep["max"][c]))
  print("valid fraction per row: " + " ".join("%.3f" % v for v in rep["row_valid_fraction"]))
  if int(rep["class_pixels"].sum()) or rep["dropped"]:
    print("class frequencies (share of the valid pixels whose label is a class id):")
    for c, name in enumerate(mc.CLASSES[:len(rep["class_pixels"])]):
      print("  %-16s %12d  %.6f" % (name, rep["class_pixels"][c], rep["class_frequency"][c]))
    if rep["dropped"]:
      print("  %d valid pixels have a label that is not a class id (0 .. %d)" % (rep["dropped"], len(rep["class_pixels"]) - 1))
  dm, ds = config_check(rep, mc)
  print("config check against %s: (mean - INPUT_MEAN) / INPUT_STD and std / INPUT_STD (about 0 and 1 when the data "
        "matches)" % config_name)
  for c, name in enumerate(chans):
    print("  %-10s %+9.4f %9.4f" % (name, dm[c], ds[c]))


def dataset_stats(a):
  import torch
  import torch.distributed as dist
  from .pipeline import shard_files
  from .sharding import Communicator, env_rank
  from .utils.args_loader import config_map
  if bool(a.data) == bool(a.scans):
    raise SystemExit("give either -d/--data (.npy range images) or --scans (raw .bin scans)")
  rank, local_rank, world = env_rank()
  torch.cuda.set_device(local_rank)
  comm = None
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    comm = Communicator()
  mc = config_map[a.config.lower()]()
  if a.data:
    all_files = sorted(glob.glob(a.data))
    if not all_files:
      raise SystemExit("no files match %s" % a.data)
    H, W = np.load(all_files[0], mmap_mode="r").shape[:2]
    st = DatasetStats(mc, H, W)
    files = shard_files(all_files, comm)
    for i in range(0, len(files), a.batch):
      st.update(np.stack([np.load(f) for f in files[i:i + a.batch]]), count_labels=not a.no_labels)
  else:
    from .dataset_convert import KITTI, ScanBatchLoader, learning_map_lut
    from .laserscan import SphericalProjector
    kitti = a.format == KITTI
    H = a.height or (64 if kitti else 32)                                    # dataset_convert.main's defaults
    fu = a.fov_up if a.fov_up is not None else (3.0 if kitti else 12.0)
    fd = a.fov_down if a.fov_down is not None else (-25.0 if kitti else -30.0)
    scans = sorted(glob.glob(a.scans))
    labels = sorted(glob.glob(a.labels)) if a.labels else None
    if labels is not None and len(labels) != len(scans):
      raise SystemExit("%d scans but %d label files" % (len(scans), len(labels)))
    lut = None
    if a.learning_map:
      import yaml
      with open(a.learning_map) as f:
        lut = learning_map_lut(yaml.safe_load(f)["learning_map"])
    scans = shard_files(scans, comm)        # both lists sorted: the same slice of each
    labels = shard_files(labels, comm) if labels is not None else None
    st = DatasetStats(mc, H, a.width)
    loader = ScanBatchLoader(a.format)
    projector = SphericalProjector(H, a.width, fu, fd, label_lut=lut)
    for i in range(0, len(scans), a.batch):
      st.update_scans(loader.load(scans[i:i + a.batch], labels[i:i + a.batch] if labels is not None else None),
                      projector, use_ring=a.ring)
  rep = st.finish(comm)
  if rank == 0:
    print_report(rep, mc, a.config)
    if a.json:
      with open(a.json, "w") as f:
        json.dump(to_json(rep), f, indent=1)
  if comm is not None:
    comm.close()
    dist.destroy_process_group()
  return rep


def build_parser():
  ap = argparse.ArgumentParser(description="per-channel mean / std, ranges, occupancy and class frequencies of a "
                                           "dataset, on the GPU")
  ap.add_argument("-d", "--data", default=None, help="glob of [H,W,5|6] .npy range images (dataset_convert's output)")
  ap.add_argument("--scans", default=None, help="glob of raw .bin scans, projected on the fly (nothing is written)")
  ap.add_argument("-n", "--config", default="squeezesegv2kitti", help="the `mc` configuration: classes, and the "
                                                                      "INPUT_MEAN / INPUT_STD to check against")
  ap.add_argument("-b", "--batch", type=int, default=64, help="frames / scans per GPU call")
  ap.add_argument("--json", default=None, help="write the statistics to this JSON file")
  ap.add_argument("--no_labels", action="store_true", help="-d: do not count the label channel (files converted "
                                                            "without label files hold 0 there)")
  ap.add_argument("--format", choices=["kitti", "nuscenes"], default="kitti")
  ap.add_argument("--labels", default=None, help="glob of .label (KITTI) / lidarseg .bin (nuScenes) files, same order")
  ap.add_argument("--learning_map", default=None, help="yaml with a `learning_map` dict (semantic-kitti.yaml)")
  ap.add_argument("--height", type=int, default=None)
  ap.add_argument("--width", type=int, default=1024)
  ap.add_argument("--fov_up", type=float, default=None)
  ap.add_argument("--fov_down", type=float, default=None)
  ap.add_argument("--ring", action="store_true", help="nuScenes: rows from the ring index (do_range_projection_ring)")
  return ap


def main(argv=None):
  return dataset_stats(build_parser().parse_args(argv))


if __name__ == "__main__":
  main()
