#!/usr/bin/env python
"""Cost of calibrated confidence (csrc/calibration.cu) at the benchmark shape: SqueezeSegV2-KITTI 64 x 2048 (random init
+ randomised BN), B = 32 frames, NC = 20; the logits of the forward (335 MB, more than the 126 MB of L2) are the input
of the pixel kernels.

Kernel times: CUDA events around --steps back-to-back calls, median of --reps repetitions:
  confidence        pcls_confidence, logits mode at T = 1.5, conf only:     NC*4 + 1 B read, 4 B written per pixel
  confidence_probs  the same with out_probs:                               + NC*4 B written per pixel
  nll64 / nll2      pcls_temperature_nll with 64 / 2 temperatures:         NC*4 + 4 B read per pixel; n_temps * NC
                    expf per counted pixel, against the MUFU exp2 rate (16 results per clock per SM, the CUDA C
                    Programming Guide's throughput table for base-2 exponentials) at the card's maximum SM clock
  reliability       pcls_reliability_update over the 4.2 M pixels:         12 B read per pixel (four input sets rotated,
                    200 MB, so that the inputs do not stay in L2)
  point_confidence  pcls_point_confidence on 16 scans of 115-125 k points: 12 B read + a 4 B gather + 4 B written per point
The HBM peak is bench.py's.  Eval steps (ms per 32-frame step, Evaluator.update on device-resident frames, alternated):
plain, --calibration (T = 1.5) and --fit_temperature (64-point grid).

    python tools/calibration_bench.py [--steps 20] [--reps 3] [--out profiles/calibration_bench_b200.json]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MUFU_EX2_PER_CLK_PER_SM = 16


def gpu_info():
  """Card name, power limit and maximum SM clock, read-only query."""
  try:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, timeout=30)
    name, power, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit_W": float(power), "max_sm_clock_MHz": float(clk)}
  except Exception as e:  # the numbers are still reported, marked as unattributed
    return {"name": None, "power_limit_W": None, "max_sm_clock_MHz": None, "error": str(e)}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--reps", type=int, default=3)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("calibration_bench: no CUDA device (there is no CPU fallback)")
  from bench import measured_peaks
  from pclsegmentation_b200 import _lib
  from pclsegmentation_b200.calibration import Calibration, inv_temperature
  from pclsegmentation_b200.laserscan import SphericalProjector
  from pclsegmentation_b200.pipeline import Evaluator
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.util import synth_range_images, synth_scan
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  info = gpu_info()
  peaks = measured_peaks()
  lib = _lib.load()
  s = torch.cuda.current_stream().cuda_stream
  B, H, W = 32, 64, 2048
  rng = np.random.default_rng(2026)
  mc = config_map["squeezesegv2kitti"]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(1)
  NC, none = mc.NUM_CLASS, mc.CLASSES.index("None")
  frames = [torch.from_numpy(synth_range_images(rng, B, H, W, channels=6, num_classes=NC)).to(dev) for _ in range(2)]
  fwd = model.forward_device(frames[0], None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_logits=True)
  logits = fwd["logits"]
  px_n = B * H * W
  label = torch.from_numpy(frames[0][..., 5].cpu().numpy().astype(np.int32)).to(dev)
  mask = (frames[0][..., 4] > 0).to(torch.uint8)
  counted = int(((label >= 0) & (label < NC) & (label != none)).sum().item())
  conf = torch.empty(px_n, dtype=torch.float32, device=dev)
  probs = torch.empty((px_n, NC), dtype=torch.float32, device=dev)
  grid = Calibration(fit=True).grid_temperatures()
  inv64 = (ctypes.c_float * 64)(*[inv_temperature(T) for T in grid])
  inv2 = (ctypes.c_float * 2)(1.0, inv_temperature(1.5))
  acc = torch.zeros(64, dtype=torch.float64, device=dev)
  cnt = torch.zeros(1, dtype=torch.int64, device=dev)
  rel_sets = [(torch.rand(px_n, device=dev), torch.randint(0, NC, (px_n,), dtype=torch.int32, device=dev),
               torch.randint(0, NC, (px_n,), dtype=torch.int32, device=dev)) for _ in range(4)]
  bins = [torch.zeros(15, dtype=t, device=dev) for t in (torch.int64, torch.int64, torch.float64)]
  # 16 scans for the point gather: projection outputs, random point labels, forward-sized probabilities
  sizes = rng.integers(115000, 125001, 16)
  pts = torch.from_numpy(np.concatenate([synth_scan(rng, int(n)) for n in sizes])).to(dev)
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).to(dev)
  proj = SphericalProjector(H, W, 3.0, -25.0).project(pts, offsets, empty_fill=0.0, want_point_outputs=True)
  total = int(sizes.sum())
  plab = torch.randint(0, NC, (total,), dtype=torch.int32, device=dev)
  pprobs = torch.rand((16, H, W, NC), device=dev)
  pconf = torch.empty(total, dtype=torch.float32, device=dev)

  def chk(rc, what):
    _lib.check(rc, what)

  kernels = {
    "confidence": (lambda i: chk(lib.pcls_confidence(logits.data_ptr(), None, mask.data_ptr(), px_n, NC,
                                                     inv_temperature(1.5), None, conf.data_ptr(), None, s), "conf"),
                   px_n * (NC * 4 + 1 + 4)),
    "confidence_probs": (lambda i: chk(lib.pcls_confidence(logits.data_ptr(), None, mask.data_ptr(), px_n, NC,
                                                           inv_temperature(1.5), probs.data_ptr(), conf.data_ptr(), None,
                                                           s), "conf"), px_n * (2 * NC * 4 + 1 + 4)),
    "nll64": (lambda i: chk(lib.pcls_temperature_nll(logits.data_ptr(), label.data_ptr(), px_n, NC, none, 64, inv64,
                                                     acc.data_ptr(), cnt.data_ptr(), s), "nll"), px_n * (NC * 4 + 4)),
    "nll2": (lambda i: chk(lib.pcls_temperature_nll(logits.data_ptr(), label.data_ptr(), px_n, NC, none, 2, inv2,
                                                    acc.data_ptr(), cnt.data_ptr(), s), "nll"), px_n * (NC * 4 + 4)),
    "reliability": (lambda i: chk(lib.pcls_reliability_update(rel_sets[i % 4][0].data_ptr(), rel_sets[i % 4][1].data_ptr(),
                                                              rel_sets[i % 4][2].data_ptr(), px_n, NC, none, 15,
                                                              bins[0].data_ptr(), bins[1].data_ptr(), bins[2].data_ptr(),
                                                              s), "rel"), px_n * 12),
    "point_confidence": (lambda i: chk(lib.pcls_point_confidence(pprobs.data_ptr(), offsets.data_ptr(), 16, H, W, total,
                                                                 proj["proj_x"].data_ptr(), proj["proj_y"].data_ptr(),
                                                                 plab.data_ptr(), NC, pconf.data_ptr(), s), "pc"),
                         total * 20),
  }

  def timed(fn):
    for i in range(3):
      fn(i)
    torch.cuda.synchronize()
    reps = []
    for _ in range(a.reps):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for i in range(a.steps):
        fn(i)
      e1.record()
      torch.cuda.synchronize()
      reps.append(e0.elapsed_time(e1) / a.steps)
    return reps

  clk = info.get("max_sm_clock_MHz")
  props = torch.cuda.get_device_properties(0)
  exp_rate = props.multi_processor_count * MUFU_EX2_PER_CLK_PER_SM * clk * 1e6 if clk else None
  kern = {}
  for name, (fn, by) in kernels.items():
    reps = timed(fn)
    ms = statistics.median(reps)
    k = {"ms": ms, "ms_reps": reps, "algorithmic_bytes": by, "GBps": by / (ms / 1e3) / 1e9,
         "frac_of_hbm_peak": by / (ms / 1e3) / 1e9 / peaks["hbm_gbs"]}
    if name.startswith("nll"):
      nt = 64 if name == "nll64" else 2
      exps = counted * nt * NC
      k.update(exps=exps, exps_per_s=exps / (ms / 1e3),
               frac_of_mufu_exp_rate=exps / (ms / 1e3) / exp_rate if exp_rate else None)
    kern[name] = k

  # eval steps: plain, --calibration, --fit_temperature, alternated
  evs = {"plain": Evaluator(model), "calibration": Evaluator(model, calibration=Calibration(temperature=1.5)),
         "fit_temperature": Evaluator(model, calibration=Calibration(temperature=1.5, fit=True))}
  steps = {k: [] for k in evs}
  for ev in evs.values():
    for i in range(2):
      ev.update(frames[i % 2])
  torch.cuda.synchronize()
  for _ in range(a.reps):
    for name, ev in evs.items():
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for i in range(a.steps):
        ev.update(frames[i % 2])
      e1.record()
      torch.cuda.synchronize()
      steps[name].append(e0.elapsed_time(e1) / a.steps)
  report = {"tool": "tools/calibration_bench.py", "gpu": info, "network": "squeezesegv2", "config": "squeezesegv2kitti",
            "B": B, "H": H, "W": W, "num_classes": NC, "counted_pixels": counted, "scan_points": total,
            "steps": a.steps, "reps": a.reps, "peak_hbm_GBps": peaks["hbm_gbs"], "peak_source": peaks["source"],
            "mufu_exp2_rate_per_s": exp_rate,
            "mufu_rate_source": "%d SMs x %d exp2 results per clock per SM (CUDA C Programming Guide, arithmetic "
                                "instruction throughput) x the maximum SM clock from nvidia-smi"
                                % (props.multi_processor_count, MUFU_EX2_PER_CLK_PER_SM),
            "kernels": kern, "eval_step_ms": {k: statistics.median(v) for k, v in steps.items()},
            "eval_step_ms_reps": steps}
  print(json.dumps(report))
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump(report, f, indent=1)


if __name__ == "__main__":
  main()
