#!/usr/bin/env python
"""bench.py - headline benchmark of the B200 inference hot path.

Metric (BASELINE.json): range-image frames/sec (SqueezeSegV2, 64x2048), plus p50 latency.
A "step" is one forward of the hot path over one batch of synthetic range images:
input stage (mask / normalise, fused) -> SqueezeSegV2 -> softmax/argmax/mask head -> predictions (+ probabilities).

    python bench.py --gpus N --steps K --warmup W            # this implementation (CUDA, one rank per GPU)
    python bench.py --impl reference --steps K --warmup W    # CPU restatement of the reference graph (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # + what the last timed step returned, as DIR/*.npy

Prints ONE JSON line on rank 0.  `value` = whole-job frames/s with inputs resident in HBM; `e2e` = the same metric
through the reference-facing call `model([lidar, mask])` with HOST (pinned) buffers, H2D + D2H inside the timed
region.  `roofline` describes the kernel that takes the largest share of the step (per-op CUDA-event timing inside
this process); `cpu_baseline` times the oracle (torch-CPU fp32 restatement of the reference graph) on the host cores.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
  # name: (model, config factory name, H, W, per-GPU batch)
  "squeezesegv2_kitti_64x2048_b32": ("squeezesegv2", "squeezesegv2kitti", 64, 2048, 32),
  "darknet21_kitti_64x2048_b32": ("darknet21", "darknet53kitti", 64, 2048, 32),
  "darknet53_kitti_64x2048_b16": ("darknet53", "darknet53kitti", 64, 2048, 16),
  "darknet53_kitti_64x2048_b64": ("darknet53", "darknet53kitti", 64, 2048, 64),
  "squeezesegv2_nuscenes_32x1024_b32": ("squeezesegv2", "squeezesegv2nuscenes", 32, 1024, 32),
}
DEFAULT_WORKLOAD = "squeezesegv2_kitti_64x2048_b32"
PROJECTION_WORKLOADS = ("projection_kitti_64x2048_b64", "darknet53_projection_64x2048_b64")


def make_config(workload):
  from pclsegmentation_b200.utils.args_loader import config_map
  model_name, cfg_name, H, W, B = WORKLOADS[workload]
  mc = config_map[cfg_name]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  if model_name == "darknet21":
    mc.NUM_LAYERS = 21  # config 3: Darknet21 + KITTI classes / mean / std (there is no darknet21kitti factory)
  return model_name, mc, B


def synth_raw(seed, B, H, W):
  """SURVEY.md §8(d) config 2 synthetic RAW range images [B,H,W,5] float32 (x,y,z,intensity,depth)."""
  sys.path.insert(0, os.path.join(ROOT, "tests"))
  from tests.util import synth_range_images
  return synth_range_images(np.random.default_rng(seed), B, H, W, valid_rate=0.78, channels=5)


class ClockSampler:
  """Samples nvidia-smi clocks / throttle reasons during the timed region."""
  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
       "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
       "clocks_event_reasons.sw_power_cap")

  def __init__(self, gpu_index):
    self.gpu = gpu_index
    self.rows = []
    self.proc = None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                   stderr=subprocess.DEVNULL, text=True)
      self.t = threading.Thread(target=self._read, daemon=True)
      self.t.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append(line.strip())

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      f = [x.strip() for x in r.split(",")]
      if len(f) < 9:
        continue
      try:
        sm.append(float(f[1]))
        mx.append(float(f[2]))
      except ValueError:
        continue
      for n, v in zip(names, f[5:9]):
        if v.lower().startswith("active"):
          reasons.add(n)
    return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(p):
    d = json.load(open(p))
    return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained",
            d["bf16_tflops"]), "source": "measured (MEASURED_PEAKS.json)"}
  return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def cpu_reference_forward(model_name, mc, model, lidar, mask):
  from oracle import nn as onn
  arch = "squeezesegv2" if model_name == "squeezesegv2" else "darknet"
  return onn.forward(arch, model.variables, lidar, mask, mc.CLASSES.index("None"),
                     num_layers=getattr(mc, "NUM_LAYERS", 53), output_stride=getattr(mc, "OUTPUT_STRIDE", 16))


def time_cpu_baseline(model_name, mc, model, raw, budget_s=12.0, max_frames=256):
  """Oracle port (torch-CPU fp32 restatement of the reference graph incl. input stage + head) on all host cores."""
  import torch
  from oracle import nn as onn
  cores = os.cpu_count() or 1
  torch.set_num_threads(cores)
  none = mc.CLASSES.index("None")
  frames, t0 = 0, time.perf_counter()
  while frames < max_frames and (frames < 1 or time.perf_counter() - t0 < budget_s):
    f = raw[frames % raw.shape[0]]
    sample = np.concatenate([f, np.zeros(f.shape[:2] + (1,), np.float32)], -1)
    lidar, mask, _ = onn.input_stage(sample, mc.INPUT_MEAN, mc.INPUT_STD, none)
    cpu_reference_forward(model_name, mc, model, lidar[None], mask[None])
    frames += 1
  dt = time.perf_counter() - t0
  return {"value": frames / dt, "unit": "frames/s", "cores": cores, "kind": "port",
          "sample": "%d frame(s) of the same %dx%d workload, batch 1, torch-CPU fp32 restatement of the reference "
                    "graph (TensorFlow 2.9.1 not installable here), %.1f s" % (frames, mc.ZENITH_LEVEL,
                                                                               mc.AZIMUTH_LEVEL, dt)}


def run_reference(args):
  """--impl reference: the reference's CPU path.  TensorFlow is absent from the image, so this is the oracle port
  (same graph, same semantics) on all host threads; each step is a bounded sample of the workload."""
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  import torch
  from oracle import nn as onn
  from pclsegmentation_b200.utils.args_loader import model_map
  model_name, mc, B = make_config(args.workload)
  model = model_map[model_name](mc)
  model.randomize_batch_norm(1)
  cores = os.cpu_count() or 1
  torch.set_num_threads(cores)
  frames_per_step = args.ref_frames
  raw = synth_raw(1234, frames_per_step, mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL)
  none = mc.CLASSES.index("None")

  def step():
    lid, msk = [], []
    for f in raw:
      sample = np.concatenate([f, np.zeros(f.shape[:2] + (1,), np.float32)], -1)
      l, m, _ = onn.input_stage(sample, mc.INPUT_MEAN, mc.INPUT_STD, none)
      lid.append(l)
      msk.append(m)
    cpu_reference_forward(model_name, mc, model, np.stack(lid), np.stack(msk))

  for _ in range(args.warmup):
    step()
  lat = []
  t0 = time.perf_counter()
  for _ in range(args.steps):
    t1 = time.perf_counter()
    step()
    lat.append(time.perf_counter() - t1)
  dt = time.perf_counter() - t0
  value = frames_per_step * args.steps / dt
  sample = "%d frame(s)/step of %s (bounded sample of the per-GPU batch %d), oracle port on %d host threads" % (
      frames_per_step, args.workload, B, cores)
  print(json.dumps({
    "impl": "reference", "metric": "range-image frames/sec (SqueezeSegV2, 64x2048)" if "squeezesegv2_kitti" in args.workload
    else "range-image frames/sec", "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
    "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
    "vs_baseline": None, "dtype": "f32", "data": "synthetic",
    "config": {"workload": args.workload, "frames_per_step": frames_per_step},
    "p50_latency_ms": 1e3 * statistics.median(lat),
    "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
    "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    "gpu_launches": 0}))


class Ranks:
  """torch.distributed plumbing of one bench process (one rank per GPU)."""

  def __init__(self):
    import torch
    import torch.distributed as dist
    self.torch, self.dist = torch, dist
    self.rank, self.local_rank, self.world = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), \
        int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
      raise SystemExit("bench.py: no CUDA device - this implementation has no CPU fallback (use --impl reference "
                       "for the CPU baseline)")
    torch.cuda.set_device(self.local_rank)
    self.dev = torch.device("cuda", self.local_rank)
    if self.world > 1:
      dist.init_process_group("nccl", device_id=self.dev)

  def barrier(self):
    if self.world > 1:
      self.dist.barrier()
    self.torch.cuda.synchronize()

  def max_over_ranks(self, v):
    t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
    if self.world > 1:
      self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
    return float(t.item())

  def close(self):
    if self.world > 1:
      self.dist.destroy_process_group()


def timed_steps(rk, step, steps, warmup):
  """`warmup` untimed steps, then exactly `steps` steps bracketed by barrier + synchronize on both sides, timed with CUDA
  events on the launching stream; returns (max-over-ranks total ms, per-step latencies of this rank, clocks of rank 0)."""
  torch = rk.torch
  for i in range(max(warmup, 3)):
    step(i)
  rk.barrier()
  sampler = ClockSampler(rk.local_rank)
  if rk.rank == 0:
    sampler.start()
    time.sleep(0.3)
  ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
  rk.barrier()
  ev[0].record()
  for i in range(steps):
    step(i)
    ev[i + 1].record()
  rk.barrier()
  total_ms = ev[0].elapsed_time(ev[-1])
  lat = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
  clocks = sampler.stop() if rk.rank == 0 else None
  return rk.max_over_ranks(total_ms), lat, clocks


DUMP_BYTES = 60 * 10 ** 6   # --dump-outputs writes at most this many bytes


def dump_outputs(out_dir, res):
  """--dump-outputs: writes what one forward returned (`res`: predictions [B,H,W] int32, probabilities [B,H,W,NC]
  float32) as out_dir/<name>.npy.  The pixels are a fixed seeded sample (every pixel when they all fit in DUMP_BYTES),
  the same for every build of the project, so that two builds can be compared file by file:
    pixel_index.npy    float64 [n]     flat index of the pixel into [B,H,W], ascending
    predictions.npy    float32 [n]     class label
    probabilities.npy  float32 [n,NC]"""
  import torch
  preds = res["predictions"].reshape(-1)
  probs = res["probabilities"].reshape(preds.numel(), -1)
  n = min(preds.numel(), (DUMP_BYTES - 3 * 128) // (8 + 4 + 4 * probs.shape[1]))   # 128: .npy header
  idx = np.sort(np.random.default_rng(0).choice(preds.numel(), n, replace=False))
  sel = torch.from_numpy(idx).to(preds.device)
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
  np.save(os.path.join(out_dir, "predictions.npy"), preds[sel].cpu().numpy().astype(np.float32))
  np.save(os.path.join(out_dir, "probabilities.npy"), probs[sel].cpu().numpy().astype(np.float32))


def op_roofline(lib, model, mc, sub, pb, outs, peaks, step_ms, B, op_table_path=None, workload=""):
  """Per-op CUDA-event table at the benchmarked batch -> roofline of the op with the largest share + whole-step totals."""
  import torch
  from pclsegmentation_b200 import _lib
  net = model._net
  n_ops = lib.pcls_net_num_ops(net)
  ms = (ctypes.c_float * n_ops)()
  acc = np.zeros(n_ops)
  mean_p = (ctypes.c_double * 5)(*mc.INPUT_MEAN.reshape(-1))
  std_p = (ctypes.c_double * 5)(*mc.INPUT_STD.reshape(-1))
  reps = 5 if pb * mc.ZENITH_LEVEL * mc.AZIMUTH_LEVEL <= 32 * 64 * 2048 and "darknet" not in workload else 2
  for r in range(reps + 1):
    _lib.check(lib.pcls_net_profile_ops(net, sub.data_ptr(), 5, None, mean_p, std_p, pb, None,
                                        outs["probabilities"].data_ptr(), outs["predictions"].data_ptr(), ms,
                                        torch.cuda.current_stream().cuda_stream), "pcls_net_profile_ops")
    if r:
      acc += np.array(list(ms))
  acc /= reps
  table = []
  tot_by = tot_fl = 0
  for i in range(n_ops):
    name = ctypes.create_string_buffer(64)
    fam, fl, by = ctypes.c_int(), ctypes.c_int64(), ctypes.c_int64()
    lib.pcls_net_op_info(net, i, name, ctypes.byref(fam), ctypes.byref(fl), ctypes.byref(by))
    tot_by += by.value
    tot_fl += fl.value
    t_s = acc[i] / 1e3
    gbs = by.value * pb / t_s / 1e9 if t_s > 0 else 0.0
    tfs = fl.value * pb / t_s / 1e12 if t_s > 0 else 0.0
    ai = fl.value / max(by.value, 1)
    bound = "tensor" if (fam.value == 1 and ai > peaks["tflops_sustained"] * 1e3 / peaks["hbm_gbs"]) else "hbm"
    table.append({"op": name.value.decode(), "ms": float(acc[i]), "share": 0.0, "GB/s": gbs, "TFLOP/s": tfs,
                  "bound": bound, "family": "tcgen05" if fam.value else "cuda-core",
                  "frac": (tfs / peaks["tflops_sustained"]) if bound == "tensor" else gbs / peaks["hbm_gbs"],
                  "algorithmic_bytes_per_frame": by.value, "flops_per_frame": fl.value})
  tot = sum(r["ms"] for r in table)
  for r in table:
    r["share"] = r["ms"] / tot if tot else 0.0
  top = max(table, key=lambda r: r["ms"])
  if top["bound"] == "tensor":
    roof = {"bound": "tensor", "achieved": top["TFLOP/s"], "peak": peaks["tflops_sustained"], "unit": "TFLOP/s"}
  else:
    roof = {"bound": "hbm", "achieved": top["GB/s"], "peak": peaks["hbm_gbs"], "unit": "GB/s"}
  traffic = None
  for tname in ("ncu_traffic_r2.json", "ncu_traffic_r1.json"):
    tpath = os.path.join(ROOT, "profiles", tname)
    if os.path.exists(tpath):  # DRAM bytes per launch of this kernel from the committed ncu --set full capture (same batch)
      t = json.load(open(tpath)).get(top["op"])
      if t and t.get("batch") == pb:
        traffic = t["dram_read_bytes"] + t["dram_write_bytes"]
        break
  roof.update(frac=roof["achieved"] / roof["peak"], traffic=traffic, kernel=top["op"], share_of_step=top["share"],
              peak_source=peaks["source"], batch_profiled=pb,
              algorithmic_bytes_per_launch=top["algorithmic_bytes_per_frame"] * pb if roof["unit"] == "GB/s" else None,
              flops_per_launch=top["flops_per_frame"] * pb,
              ops_above_1pct_below_half=[{"op": r["op"], "share": round(r["share"], 4), "frac": round(r["frac"], 3)}
                                         for r in table if r["share"] > 0.01 and r["frac"] < 0.5])
  step_s = step_ms / 1e3
  whole = {"algorithmic_GB_per_frame": tot_by / 1e9, "GFLOP_per_frame": tot_fl / 1e9,
           "achieved_GB/s": tot_by * B / step_s / 1e9, "achieved_TFLOP/s": tot_fl * B / step_s / 1e12,
           "frac_of_hbm_peak": tot_by * B / step_s / 1e9 / peaks["hbm_gbs"],
           "frac_of_tensor_peak": tot_fl * B / step_s / 1e12 / peaks["tflops_sustained"]}
  if op_table_path:
    os.makedirs(os.path.dirname(os.path.abspath(op_table_path)), exist_ok=True)
    with open(op_table_path, "w") as f:
      json.dump({"workload": workload, "batch": pb, "ops": table, "whole_step": whole}, f, indent=1)
  return roof, whole


def build_model(workload, args, batch=None):
  from pclsegmentation_b200.utils.args_loader import model_map
  model_name, mc, B = make_config(workload)
  if batch:
    B = batch
  model = model_map[model_name](mc)      # Keras-default init (glorot, seed 0) ...
  model.randomize_batch_norm(1)          # ... + randomised BN statistics so the folding is exercised
  for k, v in (("conv_impl", args.conv_impl), ("use_graph", args.use_graph), ("micro_batch", args.micro_batch)):
    if v is not None:
      model.set_option(k, v)
  for kv in args.opt:                      # A/B switches of the library (pcls_net_set_option), e.g. --opt tc_vstream=1
    k, v = kv.split("=")
    model.set_option(k, int(v))
  return model_name, mc, model, B


def resident_inputs(rk, B, H, W, nbuf):
  """`nbuf` distinct raw batches resident in HBM (rotated, so consecutive steps never see the same input)."""
  raw_host = [synth_raw(1234 + 97 * rk.rank + i, B, H, W) for i in range(nbuf)]
  return raw_host, [rk.torch.from_numpy(r).to(rk.dev) for r in raw_host]


def run_extra_workload(rk, args, workload, steps, peaks):
  """One more BASELINE configuration measured inside the same bench process (device-resident inputs, same timing
  rules); returns the entry of the line's `extra_workloads` array."""
  torch = rk.torch
  from pclsegmentation_b200 import _lib
  lib = _lib.load()
  if workload in PROJECTION_WORKLOADS:
    return projection_entry(rk, args, workload, steps, peaks)
  model_name, mc, model, B = build_model(workload, args)
  H, W, NC = mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL, mc.NUM_CLASS
  nbuf = 2 if B * H * W * 20 > 300e6 else 4
  raw_host, raw_dev = resident_inputs(rk, B, H, W, nbuf)
  outs = {"predictions": torch.empty((B, H, W), dtype=torch.int32, device=rk.dev),
          "probabilities": torch.empty((B, H, W, NC), dtype=torch.float32, device=rk.dev)}
  step = lambda i: model.forward_device(raw_dev[i % nbuf], None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD,
                                        want_probabilities=True, out=outs)
  total_ms, lat, clocks = timed_steps(rk, step, steps, 3)
  entry = {"workload": workload, "metric": "range-image frames/sec", "value": rk.world * B * steps / (total_ms / 1e3),
           "unit": "frames/s", "n_gpus": rk.world, "steps": steps, "warmup": 3, "ms_per_step": total_ms / steps,
           "per_gpu_batch": B, "H": H, "W": W, "dtype": "f16 storage / f32 accumulate", "clocks": clocks,
           "p50_latency_ms": statistics.median(lat)}
  if rk.rank == 0:
    roof, whole = op_roofline(lib, model, mc, raw_dev[0], B, outs, peaks, total_ms / steps, B, workload=workload,
                              op_table_path=(os.path.join(os.path.dirname(os.path.abspath(args.op_table)),
                                                          "optable_%s.json" % workload) if args.op_table else None))
    entry.update(roofline=roof, whole_step=whole)
  model._release()
  del raw_dev, outs
  torch.cuda.empty_cache()
  return entry


EVAL_CLASS_HIST = [0.35, 0.08, 0.20, 0.02, 0.20, 0.01, 0.01, 0.10, 0.02, 0.01]   # synthetic: Road ... Bus (None = invalid px)


def synth_eval_chunk(torch, dev, chunk_id, n, H, W):
  """BASELINE config 5 synthetic val frames [n,H,W,6] f32 (x,y,z,intensity,depth,label), generated ON the device from a
  seed that depends only on the global chunk index, so every rank (and rank 0's single-GPU recomputation) sees
  identical frames: valid ~ Bernoulli(0.60), depth ~ U(2,80), direction from the pixel centre (fov 10 / -30),
  labels ~ Categorical(EVAL_CLASS_HIST); invalid pixels all-zero."""
  g = torch.Generator(device=dev)
  g.manual_seed(90000 + chunk_id)
  valid = torch.rand((n, H, W), generator=g, device=dev) < 0.60
  depth = 2.0 + 78.0 * torch.rand((n, H, W), generator=g, device=dev)
  inten = 0.99 * torch.rand((n, H, W), generator=g, device=dev)
  hist = torch.tensor(EVAL_CLASS_HIST, device=dev)
  label = torch.multinomial(hist, n * H * W, replacement=True, generator=g).reshape(n, H, W).to(torch.float32)
  pitch = torch.deg2rad(10.0 - 40.0 * (torch.arange(H, device=dev) + 0.5) / H).reshape(1, H, 1)
  yaw = (np.pi - 2 * np.pi * (torch.arange(W, device=dev) + 0.5) / W).reshape(1, 1, W)
  x = depth * torch.cos(pitch) * torch.cos(yaw)
  y = depth * torch.cos(pitch) * torch.sin(yaw)
  z = depth * torch.sin(pitch) * torch.ones_like(yaw)
  img = torch.stack([x, y, z, inten, depth, label], -1) * valid[..., None]
  return img.to(torch.float32).contiguous()


def run_eval_leg(rk, args, frames_per_rank=1024, chunk=32):
  """BASELINE config 5 (pcl_segmentation/eval.py:41-58 sharded): SqueezeSegV2, nuScenes config (32x1024, NC 11), a
  synthetic val split of `frames_per_rank` x world frames sharded contiguously over the ranks; every rank runs
  forward -> head -> confusion update per batch on its shard, then ONE ncclAllReduce(int64) of the [NC,NC] matrix
  (pcls_confusion_allreduce).  Rank 0 then recomputes the matrix alone over ALL frames and with np.bincount on the
  host, and reports whether the three are identical."""
  torch = rk.torch
  from pclsegmentation_b200 import _lib
  from pclsegmentation_b200.pipeline import Evaluator
  from pclsegmentation_b200.sharding import Communicator, shard_range
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  lib = _lib.load()
  mc = config_map["squeezesegv2nuscenes"]()
  H, W, NC = mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL, mc.NUM_CLASS
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(1)
  comm = Communicator() if rk.world > 1 else None
  n_total = frames_per_rank * rk.world
  lo, hi = shard_range(n_total // chunk, rk.rank, rk.world)          # shards of whole chunks
  data = [synth_eval_chunk(torch, rk.dev, c, chunk, H, W) for c in range(lo, hi)]   # resident in HBM
  ev = Evaluator(model, comm)
  ev.update(data[0])                                                    # warm-up (graph capture, NCCL communicator)
  if comm is not None:
    ev.miou_tracker.allreduce(comm)
  ev.miou_tracker.reset_states()
  rk.barrier()
  e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
  e0.record()
  for d in data:
    ev.update(d)
  e1.record()
  if comm is not None:
    ev.miou_tracker.allreduce(comm)
  e2.record()
  rk.barrier()
  total_ms = rk.max_over_ranks(e0.elapsed_time(e2))
  cm = ev.miou_tracker.total_cm.clone()
  # the collective alone (all ranks arrive together): mean of 20 all-reduces of a scratch matrix
  ar_us = None
  if comm is not None:
    scratch = torch.ones((NC, NC), dtype=torch.int64, device=rk.dev)
    rk.barrier()
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a0.record()
    for _ in range(20):
      comm.allreduce_confusion(scratch)
    a1.record()
    torch.cuda.synchronize()
    ar_us = rk.max_over_ranks(a0.elapsed_time(a1) / 20 * 1e3)
    assert int(scratch[0, 0].item()) == rk.world ** 20
  same_everywhere = True
  if rk.world > 1:
    cm0 = cm.clone()
    rk.dist.broadcast(cm0, src=0)
    same = torch.tensor([1 if torch.equal(cm, cm0) else 0], device=rk.dev)
    rk.dist.all_reduce(same, op=rk.dist.ReduceOp.MIN)
    same_everywhere = bool(same.item())
  out = None
  if rk.rank == 0:
    solo = Evaluator(model, None)
    cm_np = np.zeros((NC, NC), np.int64)
    for c in range(n_total // chunk):
      d = data[c - lo] if lo <= c < hi else synth_eval_chunk(torch, rk.dev, c, chunk, H, W)
      pred, label = solo.update(d, return_label=True)
      idx = label.cpu().numpy().astype(np.int64).ravel() * NC + pred.cpu().numpy().astype(np.int64).ravel()
      cm_np += np.bincount(idx, minlength=NC * NC).reshape(NC, NC)
    cm_solo = solo.miou_tracker.total_cm
    from pclsegmentation_b200.utils.util import confusion_matrix_to_iou_recall_precision
    iou, _, _ = confusion_matrix_to_iou_recall_precision(cm)
    out = {"workload": "squeezesegv2_nuscenes_32x1024 eval: forward + head + confusion update per batch of %d, one "
                       "ncclAllReduce(int64 [%d,%d])" % (chunk, NC, NC),
           "frames": n_total, "frames_per_rank": frames_per_rank, "frames_per_s": n_total / (total_ms / 1e3),
           "ms_total": total_ms, "nranks": rk.world, "allreduce_us": ar_us,
           "collective": "ncclAllReduce(int64, sum) via pcls_confusion_allreduce" if comm is not None else None,
           "cm_pixels": int(cm.sum().item()), "cm_expected_pixels": n_total * H * W,
           "cm_equal_single_gpu": bool(torch.equal(cm, cm_solo)), "cm_equal_numpy": bool(np.array_equal(cm.cpu().numpy(), cm_np)),
           "cm_identical_on_all_ranks": same_everywhere, "miou": float(ev.miou_tracker.result()),
           "iou_per_class": [float(v) for v in np.asarray(iou)]}
  if comm is not None:
    comm.close()
  model._release()
  del data
  torch.cuda.empty_cache()
  return out


def h2d_ceiling(rk, nbytes, reps=10):
  """What the host can feed: every rank copies `nbytes` from pinned memory to its GPU `reps` times, all ranks at once
  (plain cudaMemcpyAsync on one stream) -> GB/s per rank (slowest rank) and aggregate.  The e2e number cannot exceed
  aggregate / bytes-per-frame whatever the kernels do."""
  torch = rk.torch
  src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
  dst = torch.empty(nbytes, dtype=torch.uint8, device=rk.dev)
  dst.copy_(src, non_blocking=True)
  rk.barrier()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(reps):
    dst.copy_(src, non_blocking=True)
  b.record()
  rk.barrier()
  ms = rk.max_over_ranks(a.elapsed_time(b))
  per_rank = nbytes * reps / (ms / 1e3) / 1e9
  return {"GBps_per_rank": per_rank, "GBps_aggregate": per_rank * rk.world, "bytes_per_copy": nbytes, "reps": reps,
          "how": "pinned -> device cudaMemcpyAsync, all ranks concurrently, slowest rank"}


def run_ours(args):
  rk = Ranks()
  torch, dev, rank, world = rk.torch, rk.dev, rk.rank, rk.world
  from pclsegmentation_b200 import _lib
  lib = _lib.load()
  peaks = measured_peaks()

  model_name, mc, model, B = build_model(args.workload, args, args.batch)
  H, W, NC = mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL, mc.NUM_CLASS

  # ---- inputs: NBUF distinct raw batches resident in HBM (rotated, so consecutive steps never see the same input) ----
  NBUF = 4
  raw_host, raw_dev = resident_inputs(rk, B, H, W, NBUF)
  outs = [{"predictions": torch.empty((B, H, W), dtype=torch.int32, device=dev),
           "probabilities": torch.empty((B, H, W, NC), dtype=torch.float32, device=dev)} for _ in range(2)]

  def step(i):
    return model.forward_device(raw_dev[i % NBUF], None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD,
                                want_probabilities=True, out=outs[i % 2])

  # ---- timed region: K steps, CUDA events on the launching stream, max over ranks ----
  total_ms, lat, clocks = timed_steps(rk, step, args.steps, args.warmup)
  value = world * B * args.steps / (total_ms / 1e3)
  if args.dump_outputs and rank == 0:   # before the roofline pass below overwrites outs[0]
    dump_outputs(args.dump_outputs, outs[(args.steps - 1) % 2])

  # ---- e2e: the reference-facing call with HOST buffers (pinned), H2D + forward + D2H of the predictions ----
  # host inputs in the reference's contract (normalised [B,H,W,6] float32 + bool mask), produced untimed by the
  # library's own input-stage kernel and parked in pinned host memory
  none = mc.CLASSES.index("None")
  mean_c = (ctypes.c_double * 5)(*mc.INPUT_MEAN.reshape(-1))
  std_c = (ctypes.c_double * 5)(*mc.INPUT_STD.reshape(-1))
  host_inputs = []
  for r in raw_dev[:2]:
    lid = torch.empty((B, H, W, 6), dtype=torch.float32, device=dev)
    msk = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
    _lib.check(lib.pcls_input_stage(r.data_ptr(), 5, B * H * W, mean_c, std_c, none, lid.data_ptr(), msk.data_ptr(),
                                    None, None, 0, None, torch.cuda.current_stream().cuda_stream), "pcls_input_stage")
    host_inputs.append((lid.cpu().pin_memory(), msk.cpu().bool().pin_memory(), lid.to(torch.float16).cpu().pin_memory()))
    del lid, msk
  e2e_steps = max(3, min(args.steps, 20))

  def e2e_issue(i):
    lidar, mask, _ = host_inputs[i % 2]
    probabilities, predictions = model([lidar, mask])      # H2D (copy stream) + forward, asynchronous
    return predictions

  def e2e_issue_f16(i):
    _, mask, lidar16 = host_inputs[i % 2]
    probabilities, predictions = model([lidar16, mask])    # the same call, lidar_input held as float16 on the host
    return predictions

  raw_pinned = [torch.from_numpy(r).pin_memory() for r in raw_host[:2]]

  def e2e_issue_raw(i):
    probabilities, predictions = model.predict_raw(raw_pinned[i % 2])   # inference.py's flow: raw samples in, input stage on the device
    return predictions

  def e2e_run(n, issue, depth=3):
    # the call a user makes, pipelined: `depth` batches are in flight - batch i+2 is submitted before batch i's
    # predictions are read back, so uploads, kernels and read-backs of consecutive batches overlap; EVERY step's
    # predictions are copied to the host (predictions.numpy())
    q = [issue(i) for i in range(min(depth - 1, n))]
    for i in range(len(q), n):
      q.append(issue(i))
      q.pop(0).numpy()                                    # D2H (synchronises on the oldest batch in flight)
    while q:
      q.pop(0).numpy()

  def e2e_measure(issue, h2d_bytes):
    e2e_run(3, issue)
    rk.barrier()
    t0 = time.perf_counter()
    e2e_run(e2e_steps, issue)
    rk.barrier()
    return world * B * e2e_steps / rk.max_over_ranks(time.perf_counter() - t0)

  # Three host representations of the same frames go through the same public call.  The headline is the 16-bit one:
  # the network stores its input as 16-bit values anyway (results are bit-identical, tests/test_gpu_nets.py), and at
  # 8 ranks the box's host side (one NUMA node feeding 8 GPUs) cannot deliver 25 bytes per pixel at the kernels' rate.
  f32_bytes, f16_bytes, raw_bytes, d2h_bytes = B * H * W * (6 * 4 + 1), B * H * W * (6 * 2 + 1), B * H * W * 20, B * H * W * 4
  e2e_f32_value = e2e_measure(e2e_issue, f32_bytes)
  e2e_raw_value = e2e_measure(e2e_issue_raw, raw_bytes)
  e2e_value = e2e_measure(e2e_issue_f16, f16_bytes)
  ceiling = h2d_ceiling(rk, f32_bytes)
  agg = ceiling["GBps_aggregate"]

  def variant(v, nbytes, call):
    return {"value": v, "unit": "frames/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": d2h_bytes, "call": call,
            "h2d_GBps_aggregate_achieved": v * (nbytes / B) / 1e9, "frac_of_host_ceiling": v * (nbytes / B) / 1e9 / agg,
            "frames_per_s_at_host_ceiling": agg * 1e9 / (nbytes / B)}

  e2e = variant(e2e_value, f16_bytes,
                "model([lidar float16 [B,H,W,6], mask bool]) -> predictions.numpy(): the reference's call with lidar_input "
                "held as float16 on the host (13 B/pixel; bit-identical results to the float32 input), pinned host inputs, "
                "3 batches in flight, %d steps" % e2e_steps)
  e2e["host_h2d_ceiling"] = ceiling
  e2e["f32_contract"] = variant(e2e_f32_value, f32_bytes,
                                "model([lidar float32 [B,H,W,6], mask bool]) -> predictions.numpy() (25 B/pixel), same pipeline")
  e2e["raw_input"] = variant(e2e_raw_value, raw_bytes,
                             "model.predict_raw(raw [B,H,W,5] f32) -> predictions.numpy() (inference.py:47-78 as one call: "
                             "the input stage runs on the device, 20 B/pixel), same pipeline")
  del host_inputs

  # ---- the other BASELINE configurations, same process, same timing rules (all ranks take part) ----
  extras = []
  if not args.no_extras and args.workload == DEFAULT_WORKLOAD:
    main_bufs = (raw_dev, outs)
    for w, st in EXTRA_WORKLOADS:
      try:
        extras.append(run_extra_workload(rk, args, w, st, peaks))
      except Exception as e:  # an extra workload must never take the headline line down
        extras.append({"workload": w, "error": "%s: %s" % (type(e).__name__, e)})
  eval_leg = None
  if not args.no_eval and args.workload == DEFAULT_WORKLOAD:
    try:
      eval_leg = run_eval_leg(rk, args, frames_per_rank=args.eval_frames)
    except Exception as e:
      eval_leg = {"error": "%s: %s" % (type(e).__name__, e)}

  if rank != 0:
    rk.close()
    return

  # ---- rank 0 only: batch-1 latency, per-op roofline table, CPU baseline ----
  lat1 = []
  one = raw_dev[0][:1].contiguous()
  for i in range(25):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    model.forward_device(one, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_probabilities=True)
    b.record()
    b.synchronize()
    if i >= 5:
      lat1.append(a.elapsed_time(b))

  net = model._net
  pb = B if not args.micro_batch else min(B, args.micro_batch)   # profile at the benchmarked batch
  roof, whole = op_roofline(lib, model, mc, raw_dev[1][:pb].contiguous(), pb, outs[0], peaks, total_ms / args.steps, B,
                            op_table_path=args.op_table, workload=args.workload)

  cpu = time_cpu_baseline(model_name, mc, model, raw_host[0]) if not args.no_cpu_baseline else None
  launches = lib.pcls_net_launches_per_forward(net)
  passes = -(-B // args.micro_batch) if args.micro_batch else 1
  line = {
    "metric": "range-image frames/sec (SqueezeSegV2, 64x2048)" if args.workload == DEFAULT_WORKLOAD else
              "range-image frames/sec (%s)" % args.workload,
    "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
    "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
    "dtype": "f16 storage / f32 accumulate", "data": "synthetic",
    "config": {"workload": args.workload, "per_gpu_batch": B, "global_batch": B * world, "H": H, "W": W,
               "input": "raw [B,H,W,5] f32 resident in HBM; input stage (mask / normalise) inside pcls_net_forward (its own kernel)",
               "outputs": "predictions i32 + probabilities f32",
               "weights": "Keras-default init seed 0 + randomised BN", "l2_policy":
               "inputs rotate over %d resident batches (%.0f MB) and each step streams > 1 GB of activations, far above "
               "the 126 MB L2" % (NBUF, NBUF * B * H * W * 20 / 1e6),
               "parallelism": "dp%d (frames sharded, no data-path collective)" % world,
               "options": model.net_options},
    "p50_latency_ms": {"batch_%d" % B: statistics.median(lat), "batch_1": statistics.median(lat1) if lat1 else None},
    "clocks": clocks, "e2e": e2e, "gpu_launches": launches * passes * args.steps,
    "roofline": roof, "whole_step": whole, "cpu_baseline": cpu,
  }
  if extras:
    line["extra_workloads"] = extras
  if eval_leg is not None:
    line["eval"] = eval_leg
  print(json.dumps(line))
  rk.close()


EXTRA_WORKLOADS = [  # (workload, timed steps): BASELINE configs 3, 4 and 5's network, measured inside the default run
  ("darknet21_kitti_64x2048_b32", 10),
  ("darknet53_kitti_64x2048_b64", 5),
  ("darknet53_projection_64x2048_b64", 5),
  ("projection_kitti_64x2048_b64", 20),
  ("squeezesegv2_nuscenes_32x1024_b32", 20),
]


def projection_entry(rk, args, workload, steps, peaks):
  """BASELINE config 4 inside the default run: 64 raw scans (~120 k points each) per rank -> range images (+ Darknet53
  forward + head for the fused workload)."""
  torch = rk.torch
  from pclsegmentation_b200.laserscan import SphericalProjector
  from pclsegmentation_b200.pipeline import ScanSegmenter
  from tests.util import synth_scan
  dev = rk.dev
  B, H, W = 64, 64, 2048
  rng = np.random.default_rng(4321 + rk.rank)
  sizes = rng.integers(115000, 125001, B)
  bufs = []
  for k in range(3):  # rotate over three resident scan sets (3 x 123 MB > L2)
    bufs.append(torch.from_numpy(np.concatenate([synth_scan(rng, int(n)) for n in sizes])).to(dev))
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).to(dev)
  total = int(sizes.sum())
  fused = workload.startswith("darknet53")
  model = None
  if fused:
    _, mc, model, _ = build_model("darknet53_kitti_64x2048_b64", args)
    seg = ScanSegmenter(model, 3.0, -25.0)
    step = lambda i: seg.segment_device(bufs[i % 3], offsets)
  else:
    proj = SphericalProjector(H, W, 3.0, -25.0)
    step = lambda i: proj.project(bufs[i % 3], offsets, empty_fill=0.0)
  total_ms, lat, clocks = timed_steps(rk, step, steps, 3)
  ms = total_ms / steps
  entry = {"workload": workload, "metric": "scans/sec", "value": rk.world * B / (ms / 1e3), "unit": "scans/s",
           "n_gpus": rk.world, "steps": steps, "warmup": 3, "ms_per_step": ms, "scans_per_gpu": B, "points_per_gpu": total,
           "H": H, "W": W, "dtype": "f32/i32 (projection)" + (" + f16 net" if fused else ""), "clocks": clocks}
  if not fused:
    alg = 16 * total + B * H * W * (24 + 4)   # SURVEY.md §8(d): 16 N read + H W (6*4 + 4) written
    entry["roofline"] = {"bound": "hbm", "achieved": alg / (ms / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": alg / (ms / 1e3) / 1e9 / peaks["hbm_gbs"], "traffic": None,
                         "kernel": "project_scatter + project_resolve", "peak_source": peaks["source"],
                         "algorithmic_bytes_per_launch": alg}
  if model is not None:
    model._release()
  del bufs
  torch.cuda.empty_cache()
  return entry


def run_projection(args):
  """Side benchmarks (not the headline line): BASELINE config 4.
  projection_kitti_64x2048_b64      64 raw scans (~120 k points) -> [64,64,2048,6] range images + proj_idx
  darknet53_projection_64x2048_b64  the same projection fused with the Darknet53 forward + head (scans in, labels out)"""
  import torch
  from pclsegmentation_b200.laserscan import SphericalProjector
  from pclsegmentation_b200.pipeline import ScanSegmenter
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.util import synth_scan
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  B, H, W = (args.batch or 64), 64, 2048
  rng = np.random.default_rng(4321)
  sizes = rng.integers(115000, 125001, B)
  bufs = []
  for k in range(3):  # rotate over three resident scan sets (3 x 123 MB > L2)
    scans = np.concatenate([synth_scan(rng, int(n)) for n in sizes])
    bufs.append(torch.from_numpy(scans).to(dev))
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).to(dev)
  total = int(sizes.sum())
  fused = args.workload.startswith("darknet53")
  if fused:
    mc = config_map["darknet53kitti"]()
    mc.AZIMUTH_LEVEL = W
    model = model_map["darknet53"](mc)
    model.randomize_batch_norm(1)
    seg = ScanSegmenter(model, 3.0, -25.0)
    step = lambda i: seg.segment_device(bufs[i % 3], offsets)
  else:
    proj = SphericalProjector(H, W, 3.0, -25.0)
    step = lambda i: proj.project(bufs[i % 3], offsets, empty_fill=0.0)
  for i in range(max(args.warmup, 3)):
    step(i)
  torch.cuda.synchronize()
  sampler = ClockSampler(0)
  sampler.start()
  time.sleep(0.3)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for i in range(args.steps):
    step(i)
  e1.record()
  torch.cuda.synchronize()
  ms = e0.elapsed_time(e1) / args.steps
  clocks = sampler.stop()
  peaks = measured_peaks()
  line = {"metric": "scans/sec (%s)" % args.workload, "value": B / (ms / 1e3), "unit": "scans/s", "n_gpus": 1,
          "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f32/i32 (projection)" + (" + f16 net" if fused else ""),
          "data": "synthetic", "config": {"workload": args.workload, "scans": B, "points": total, "H": H, "W": W},
          "clocks": clocks}
  if not fused:
    alg = 16 * total + B * H * W * (24 + 4)   # SURVEY.md §8(d): 16 N read + H W (6*4 + 4) written
    line["roofline"] = {"bound": "hbm", "achieved": alg / (ms / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": alg / (ms / 1e3) / 1e9 / peaks["hbm_gbs"], "traffic": None,
                        "kernel": "project_scatter + project_resolve (+ key memset)", "peak_source": peaks["source"]}
    if not args.no_cpu_baseline:  # the oracle restatement, single thread, bounded sample
      from oracle import projection as P
      host = bufs[0][: int(offsets[4].item())].cpu().numpy()
      t0 = time.perf_counter()
      for b in range(4):
        s = host[int(offsets[b]): int(offsets[b + 1])]
        P.assemble_range_image(P.range_projection(s[:, :3], s[:, 3], H, W, 3.0, -25.0, "libm"))
      line["cpu_baseline"] = {"value": 4 / (time.perf_counter() - t0), "unit": "scans/s", "cores": 1, "kind": "port",
                              "sample": "4 scans of the same batch, numpy oracle restatement of LaserScan, 1 thread"}
  print(json.dumps(line))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS) + list(PROJECTION_WORKLOADS))
  ap.add_argument("--batch", type=int, default=None, help="override the per-GPU batch")
  ap.add_argument("--conv-impl", type=int, default=None)
  ap.add_argument("--use-graph", type=int, default=None)
  ap.add_argument("--micro-batch", type=int, default=None)
  ap.add_argument("--opt", action="append", default=[], help="library A/B switch name=value (repeatable)")
  ap.add_argument("--op-table", default=None, help="write the per-op roofline table (JSON) here")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-extras", action="store_true", help="skip the extra_workloads array (BASELINE configs 3-5)")
  ap.add_argument("--no-eval", action="store_true", help="skip the config-5 eval leg (sharded eval + NCCL all-reduce)")
  ap.add_argument("--eval-frames", type=int, default=1024, help="eval leg: synthetic val frames per rank")
  ap.add_argument("--ref-frames", type=int, default=2, help="--impl reference: frames per step (bounded sample)")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write the predictions and probabilities of the last timed step (rank 0) to DIR/*.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and (args.impl == "reference" or args.workload in PROJECTION_WORKLOADS):
    ap.error("--dump-outputs is implemented for the network workloads of --impl ours")
  if args.workload in PROJECTION_WORKLOADS:
    run_projection(args)
  elif args.impl == "reference":
    run_reference(args)
  else:
    run_ours(args)


if __name__ == "__main__":
  main()
