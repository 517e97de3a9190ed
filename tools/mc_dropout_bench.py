#!/usr/bin/env python
"""Cost of MC dropout (csrc/mc_dropout.cu) at the benchmark shape: SqueezeSegV2-KITTI 64 x 2048 (random init +
randomised BN), B = 32 frames resident in HBM, NC = 20; and Darknet21 at 64 x 2048, B = 8.

Kernel times from torch.profiler (CUDA activity, a run of its own) over --steps MC steps at T = 4:
  dropout_kernel        per site; algorithmic bytes = twice the tensor (read and written in place)
  mc_accumulate_kernel  3 * NC * 4 + 4 + 16 B per pixel (probs read, acc read + written, f64 entropy read + written)
  mc_finalize_kernel    NC * 4 + 8 + 1 B read, 4 * 4 B written per pixel (no probabilities)
The HBM peak is bench.py's.  Steps (ms per batch, CUDA events around --steps calls, median of --reps alternated
repetitions): the plain forward and forward_mc at T = 1, 4 and 8, against T x the plain step.

    python tools/mc_dropout_bench.py [--steps 10] [--reps 3] [--out profiles/mc_dropout_bench_b200.json]
    PCLS_PDL_EARLY_PX=1 python tools/mc_dropout_bench.py --out profiles/mc_dropout_bench_b200_late_pdl.json
The second run turns the early PDL trigger off (common.cuh): a dependent kernel then becomes resident only when the one
in front of it has finished, so a kernel's profiled duration holds no wait for its producer.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
  """Card name and power limit, read-only query."""
  try:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, timeout=30)
    name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_W": float(power)}
  except Exception as e:  # the numbers are still reported, marked as unattributed
    return {"name": None, "power_limit_W": None, "error": str(e)}


def workload(torch, dev, name, cfg, B, steps, reps, peaks):
  from pclsegmentation_b200.mc_dropout import MCDropout, forward_mc
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.util import synth_range_images
  H, W = 64, 2048
  mc = config_map[cfg]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  model = model_map[name](mc)
  model.randomize_batch_norm(1)
  NC = mc.NUM_CLASS
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(1), B, H, W, channels=6, num_classes=NC)).to(dev)
  mcd = {T: MCDropout(passes=T, seed=1, rate=0.5) for T in (1, 4, 8)}
  plain = lambda: model.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_probabilities=False)
  runs = {"plain": plain}
  for T in (1, 4, 8):
    runs["mc_T%d" % T] = (lambda T=T: forward_mc(model, raw, mcd[T]))
  for f in runs.values():   # warm-up: builds both nets, captures their graphs
    f()
    f()
  torch.cuda.synchronize()
  times = {k: [] for k in runs}
  for _ in range(reps):
    for k, f in runs.items():     # alternated
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(steps):
        f()
      e1.record()
      torch.cuda.synchronize()
      times[k].append(e0.elapsed_time(e1) / steps)
  step_ms = {k: statistics.median(v) for k, v in times.items()}
  # kernel times: profiler over T = 4 steps
  with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(steps):
      runs["mc_T4"]()
    torch.cuda.synchronize()
  kt = {}
  evs = [ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
  evs.sort(key=lambda ev: ev.time_range.start)   # one stream: start order is launch order (sites 0, 1, ... per pass)
  for ev in evs:
    kname = ev.name
    if "set_dropout" in kname:
      key = "set_dropout_kernel"
    elif "dropout_kernel" in kname:
      key = "dropout_kernel"
    elif "mc_accumulate" in kname:
      key = "mc_accumulate_kernel"
    elif "mc_finalize" in kname:
      key = "mc_finalize_kernel"
    else:
      continue
    kt.setdefault(key, []).append((ev.time_range.end - ev.time_range.start) / 1e3)
  px = B * H * W
  sites = model._graph.dropout_sites
  site_bytes = [2 * B * H * s.width * s.channels * 2 for s, _, _ in sites]
  kern = {}
  hbm = peaks["hbm_gbs"] * 1e9
  if "dropout_kernel" in kt:
    d = kt["dropout_kernel"]
    if len(d) != steps * 4 * len(sites):
      raise SystemExit("mc_dropout_bench: %d dropout launches, expected %d" % (len(d), steps * 4 * len(sites)))
    per_site = [statistics.median(d[i::len(sites)]) for i in range(len(sites))]
    kern["dropout"] = [{"site": k, "channels": s.channels, "width": s.width, "ms": per_site[k],
                        "bytes": site_bytes[k], "frac_of_hbm_peak": site_bytes[k] / (per_site[k] * 1e-3) / hbm}
                       for k, (s, _, _) in enumerate(sites)]
  for key, by in (("mc_accumulate_kernel", px * (3 * NC * 4 + 4 + 16)), ("mc_finalize_kernel", px * (NC * 4 + 8 + 1 + 16))):
    if key in kt:
      ms = statistics.median(kt[key])
      kern[key] = {"ms": ms, "bytes": by, "frac_of_hbm_peak": by / (ms * 1e-3) / hbm}
  model._release()
  return {"model": name, "pdl_early_px": os.environ.get("PCLS_PDL_EARLY_PX", "default (2^20)"), "config": cfg, "B": B, "H": H, "W": W, "NC": NC, "rate": 0.5, "step_ms": step_ms,
          "mc_over_T_x_plain": {T: step_ms["mc_T%d" % T] / (T * step_ms["plain"]) for T in (1, 4, 8)},
          "kernels": kern, "step_ms_reps": times}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--reps", type=int, default=3)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("mc_dropout_bench: no CUDA device (there is no CPU fallback)")
  from bench import measured_peaks
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  info = gpu_info()
  peaks = measured_peaks()
  rep = {"gpu": info, "hbm_peak_gbs": peaks["hbm_gbs"], "peak_source": peaks["source"],
         "workloads": [workload(torch, dev, "squeezesegv2", "squeezesegv2kitti", 32, a.steps, a.reps, peaks),
                       workload(torch, dev, "darknet21", "darknet21", 8, a.steps, a.reps, peaks)]}
  text = json.dumps(rep, indent=1, default=float)
  print(text)
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      f.write(text + "\n")


if __name__ == "__main__":
  main()
