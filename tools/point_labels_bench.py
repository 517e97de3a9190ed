#!/usr/bin/env python
"""Cost of per-point labels on the raw-scan path (BASELINE config 4): 64 scans of 115-125 k points at 64 x 2048, three
resident scan sets rotated as in bench.py's projection leg, SqueezeSegV2-KITTI and Darknet53-KITTI (random init +
randomised BN).

Three variants of ScanSegmenter.segment_device, alternating within the run, >= 20 timed steps each, median of three
repetitions:
  pixel  segment_device(points, offsets)                         labels per pixel (the path without point labels)
  plain  + want_point_labels=True                                each point takes its pixel's label (search 1)
  knn    + want_point_labels=True, knn=KNN()                     5 x 5 window, k 5, sigma 1, cutoff 1 m
plus the pcls_point_labels launches alone (CUDA events over 50 calls on the same batch).  Algorithmic bytes per batch,
from shapes: point pass 16 B per point (proj_x, proj_y, range read; label written), pixel pass 24 B per pixel (key and
prediction read, packed word written; the winner-range gather is not credited); the window reads come from on-chip
caches and are not credited either.  The HBM peak is bench.py's.

    python tools/point_labels_bench.py [--steps 20] [--reps 3] [--out profiles/point_labels_bench.json]
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


def gpu_info():
  """Card name and power limit, read-only query."""
  try:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return {"name": name, "power_limit": power}
  except Exception as e:  # the numbers are still reported, marked as unattributed
    return {"name": None, "power_limit": None, "error": str(e)}


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--reps", type=int, default=3)
  ap.add_argument("--kernel-calls", type=int, default=50)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("point_labels_bench: no CUDA device (there is no CPU fallback)")
  from bench import measured_peaks
  from pclsegmentation_b200 import _lib
  from pclsegmentation_b200.laserscan import SphericalProjector
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.util import synth_scan
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  peaks = measured_peaks()
  B, H, W = 64, 64, 2048
  rng = np.random.default_rng(4321)          # bench.py's projection leg
  sizes = rng.integers(115000, 125001, B)
  bufs = [torch.from_numpy(np.concatenate([synth_scan(rng, int(n)) for n in sizes])).to(dev) for _ in range(3)]
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).to(dev)
  total = int(sizes.sum())
  knn = KNN()
  point_bytes, pixel_bytes = 16 * total, 24 * B * H * W
  report = {"tool": "tools/point_labels_bench.py", "gpu": gpu_info(), "scans": B, "points": total, "H": H, "W": W,
            "steps": a.steps, "reps": a.reps, "peak_hbm_GBps": peaks["hbm_gbs"], "peak_source": peaks["source"],
            "algorithmic_bytes": {"point_pass": point_bytes, "pixel_pass": pixel_bytes}, "networks": []}

  for model_name, cfg in (("squeezesegv2", "squeezesegv2kitti"), ("darknet53", "darknet53kitti")):
    mc = config_map[cfg]()
    mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
    model = model_map[model_name](mc)
    model.randomize_batch_norm(1)
    seg = ScanSegmenter(model, 3.0, -25.0)
    variants = {
      "pixel": lambda i: seg.segment_device(bufs[i % 3], offsets),
      "plain": lambda i: seg.segment_device(bufs[i % 3], offsets, want_point_labels=True),
      "knn": lambda i: seg.segment_device(bufs[i % 3], offsets, want_point_labels=True, knn=knn),
    }
    for step in variants.values():
      for i in range(3):
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

    # the point-label launches alone, on the predictions of one forward
    res = seg.segment_device(bufs[0], offsets)
    proj = SphericalProjector(H, W, 3.0, -25.0).project(bufs[0], offsets, want_image=False, want_idx=False,
                                                        want_point_outputs=True)
    kern = {}
    lib = _lib.load()
    out = torch.empty(total, dtype=torch.int32, device=dev)
    scratch = torch.empty((B, H, W), dtype=torch.int64, device=dev)
    wt = knn.weights()
    w = (ctypes.c_float * wt.size)(*wt.tolist())
    s = torch.cuda.current_stream().cuda_stream
    for name, kk in (("plain", None), ("knn", knn)):
      # the C entry point itself with preallocated buffers: the launches, not the Python around them
      args = (res["predictions"].data_ptr(), proj["keys"].data_ptr(), offsets.data_ptr(), B, H, W, total,
              proj["proj_x"].data_ptr(), proj["proj_y"].data_ptr(), proj["unproj_range"].data_ptr(), mc.NUM_CLASS,
              mc.CLASSES.index("None"), 1 if kk is None else kk.search, 1 if kk is None else kk.k,
              None if kk is None else w, 0.0 if kk is None else kk.cutoff, -1 if kk is None else kk.ignore_index(mc),
              None if kk is None else scratch.data_ptr(), out.data_ptr(), s)
      _lib.check(lib.pcls_point_labels(*args), "pcls_point_labels")
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(a.kernel_calls):
        lib.pcls_point_labels(*args)
      e1.record()
      _lib.check(lib.pcls_point_labels(*args), "pcls_point_labels")
      torch.cuda.synchronize()
      t = e0.elapsed_time(e1) / a.kernel_calls
      by = point_bytes + (pixel_bytes if kk is not None else 0)
      kern[name] = {"ms": t, "algorithmic_bytes": by, "GBps": by / (t / 1e3) / 1e9,
                    "frac_of_hbm_peak": by / (t / 1e3) / 1e9 / peaks["hbm_gbs"]}
    entry = {"network": model_name, "config": cfg,
             "ms_per_step": {k: round(v, 4) for k, v in med.items()},
             "ms_per_step_reps": ms,
             "scans_per_s": {k: B / (v / 1e3) for k, v in med.items()},
             "overhead_vs_pixel": {k: med[k] / med["pixel"] - 1.0 for k in ("plain", "knn")},
             "point_label_launches": kern}
    report["networks"].append(entry)
    print(json.dumps(entry), flush=True)
    model._release()
    del seg, model, res, proj
    torch.cuda.empty_cache()
  print(json.dumps(report))
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump(report, f, indent=1)


if __name__ == "__main__":
  main()
