#!/usr/bin/env python
"""Cost of test-time augmentation (tta.forward_tta) at the benchmark shape: SqueezeSegV2-KITTI 64 x 2048 (random init +
randomised BN), B = 32 device-resident raw float32 frames, four input sets rotated so the inputs (4 x 100 MB) exceed L2.

Variants, alternating within the run, >= 20 timed steps each, median of three repetitions:
  plain     model.forward_device(raw, mean, std)                 the raw forward without TTA
  tta1      forward_tta(TTA(flip=False, shifts=(0,)))            identity: views + 32-frame forward + merge
  tta2      forward_tta(TTA())                                   the mirror, T = 2
  tta4      forward_tta(TTA(shifts=(0, 1024)))                   mirror x {0, W/2}, T = 4
  scan      ScanSegmenter.segment_device(want_point_labels, knn=KNN())           32 raw scans of 115-125 k points
  scan_tta  the same with tta=TTA()
Each T-view step is compared with T x plain + the two TTA kernels.  The kernel times come from a separate
torch.profiler run (CUDA activities) over the T = 2 and T = 4 steps.  Algorithmic bytes per call, from shapes:
views C x 4 B read + T x (16 + 1) B written per source pixel; merge T x NC x 4 + 1 B read + 4 B written per output pixel.
The HBM peak is bench.py's.

    python tools/tta_bench.py [--steps 20] [--reps 3] [--out profiles/tta_bench_b200.json]
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
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}
  except Exception as e:  # the numbers are still reported, marked as unattributed
    return {"name": None, "power_limit": None, "error": str(e)}


def kernel_times(prof, names):
  """{name: (calls, total device ms)} of the kernels whose name contains each of `names`."""
  out = {n: [0, 0.0] for n in names}
  for e in prof.key_averages():
    for n in names:
      if n in e.key:
        t = getattr(e, "device_time_total", None)
        if t is None:
          t = e.cuda_time_total
        out[n][0] += e.count
        out[n][1] += t / 1e3
  return out


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--reps", type=int, default=3)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("tta_bench: no CUDA device (there is no CPU fallback)")
  from bench import measured_peaks
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  from pclsegmentation_b200.tta import TTA, forward_tta
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.util import synth_range_images, synth_scan
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  peaks = measured_peaks()
  B, H, W, C = 32, 64, 2048, 6
  rng = np.random.default_rng(2026)
  sets = [torch.from_numpy(synth_range_images(rng, B, H, W, channels=C)).to(dev) for _ in range(4)]
  sizes = rng.integers(115000, 125001, B)
  scans = [torch.from_numpy(np.concatenate([synth_scan(rng, int(n)) for n in sizes])).to(dev) for _ in range(3)]
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).to(dev)

  def make_model():
    mc = config_map["squeezesegv2kitti"]()
    mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
    m = model_map["squeezesegv2"](mc)
    m.randomize_batch_norm(1)
    return mc, m

  mc, m1 = make_model()           # one model per frame count: each net is built for the batch it runs
  _, m2 = make_model()
  _, m4 = make_model()
  NC = mc.NUM_CLASS
  knn = KNN()
  seg1, seg2 = ScanSegmenter(m1, 3.0, -25.0), ScanSegmenter(m2, 3.0, -25.0)
  ttas = {1: TTA(flip=False, shifts=(0,)), 2: TTA(), 4: TTA(shifts=(0, W // 2))}
  variants = {
    "plain": lambda i: m1.forward_device(sets[i % 4], None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_probabilities=False),
    "tta1": lambda i: forward_tta(m1, sets[i % 4], ttas[1]),
    "tta2": lambda i: forward_tta(m2, sets[i % 4], ttas[2]),
    "tta4": lambda i: forward_tta(m4, sets[i % 4], ttas[4]),
    "scan": lambda i: seg1.segment_device(scans[i % 3], offsets, want_point_labels=True, knn=knn),
    "scan_tta": lambda i: seg2.segment_device(scans[i % 3], offsets, want_point_labels=True, knn=knn, tta=ttas[2]),
  }
  for step in variants.values():
    for i in range(4):
      step(i)
  torch.cuda.synchronize()
  ms = {k: [] for k in variants}
  for _ in range(a.reps):
    for name, step in variants.items():      # alternating: each repetition times every variant once
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for i in range(a.steps):
        step(i)
      e1.record()
      torch.cuda.synchronize()
      ms[name].append(e0.elapsed_time(e1) / a.steps)
  med = {k: statistics.median(v) for k, v in ms.items()}

  # kernel times in a run of their own (tracing slows the host)
  from torch.profiler import ProfilerActivity, profile
  kern = {}
  px = B * H * W
  for T in (2, 4):
    model = m2 if T == 2 else m4
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
      for i in range(a.steps):
        forward_tta(model, sets[i % 4], ttas[T])
      torch.cuda.synchronize()
    kt = kernel_times(prof, ("tta_views_kernel", "tta_merge_kernel"))
    by = {"tta_views_kernel": px * (C * 4 + T * 17), "tta_merge_kernel": px * (T * NC * 4 + 1 + 4)}
    for name, (calls, total) in kt.items():
      t = total / max(calls, 1)
      kern["%s_T%d" % (name, T)] = {"calls": calls, "ms": t, "algorithmic_bytes": by[name],
                                    "GBps": by[name] / (t / 1e3) / 1e9 if t > 0 else None,
                                    "frac_of_hbm_peak": by[name] / (t / 1e3) / 1e9 / peaks["hbm_gbs"] if t > 0 else None}
  expect = {}
  for T in (2, 4):
    k = kern["tta_views_kernel_T%d" % T]["ms"] + kern["tta_merge_kernel_T%d" % T]["ms"]
    want = T * med["plain"] + k
    expect["tta%d" % T] = {"T_x_plain_plus_kernels_ms": want, "measured_ms": med["tta%d" % T],
                           "ratio": med["tta%d" % T] / want}
  report = {"tool": "tools/tta_bench.py", "gpu": gpu_info(), "network": "squeezesegv2", "config": "squeezesegv2kitti",
            "B": B, "H": H, "W": W, "channels": C, "num_classes": NC, "scan_points": int(sizes.sum()),
            "steps": a.steps, "reps": a.reps, "peak_hbm_GBps": peaks["hbm_gbs"], "peak_source": peaks["source"],
            "ms_per_step": {k: round(v, 4) for k, v in med.items()}, "ms_per_step_reps": ms,
            "frames_per_s": {k: B / (v / 1e3) for k, v in med.items()},
            "kernels": kern, "t_view_step_vs_expected": expect}
  print(json.dumps(report))
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump(report, f, indent=1)


if __name__ == "__main__":
  main()
