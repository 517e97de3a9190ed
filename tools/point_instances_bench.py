#!/usr/bin/env python
"""Cost of instance ids on the raw-scan path: 64 synthetic scans of 115-125 k points at 64 x 2048 with planted objects
(boxes and cylinders of thing points at 5-60 m, one across the azimuth seam, plus ground and background; the generator
of tests/test_gpu_point_instances.py), labels from the planted truth.

  kernel   pcls_point_instances alone on the planted labels, default Clustering() (tau 0.5 m, 3 x 5 window, 10 points),
           CUDA events over --kernel-calls calls, --reps repetitions; plus a per-kernel split from torch.profiler (a run of
           its own).
  step     SqueezeSegV2-KITTI (random init + randomised BN) ScanSegmenter.segment_device with the k-NN vote, without and
           with instances=Clustering(), alternating, --steps timed steps per repetition; the thing points there are
           whatever the random-init network predicts.
Counts per batch from the oracle on the host: nodes (thing pixels), node pairs tested in the forward half of the window,
edges (pairs joined).  Algorithmic bytes per batch, from shapes: per pixel 40 B (key read; parent written, read by the
union, flatten and number passes, written by flatten; size written, read and written by the number pass), per node
52 B (winner's x, y, z, w and label read, node word written, read by the union pass), per point 44 B (proj_x, proj_y,
label, x, y, z, w read; stashed root written, read and rewritten; root's id gathered); window reads of neighbours and
the gathers of the point pass are not credited.  The HBM peak is bench.py's.

    python tools/point_instances_bench.py [--steps 20] [--reps 5] [--out profiles/point_instances_bench_b200.json]
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--reps", type=int, default=5)
  ap.add_argument("--kernel-calls", type=int, default=50)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("point_instances_bench: no CUDA device (there is no CPU fallback)")
  from bench import measured_peaks
  from oracle import point_instances as PI
  from pclsegmentation_b200 import _lib
  from pclsegmentation_b200.laserscan import SphericalProjector
  from pclsegmentation_b200.pipeline import KNN, Clustering, ScanSegmenter
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.test_gpu_point_instances import KITTI_THINGS, bench_scans
  from tools.point_labels_bench import gpu_info
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  peaks = measured_peaks()
  B, H, W = 64, 64, 2048
  sizes, scans, labels, _ = bench_scans(B)
  total = int(sizes.sum())
  offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  pts = torch.from_numpy(np.concatenate(scans)).to(dev)
  lab = torch.from_numpy(np.concatenate(labels)).to(dev)
  offsets = torch.from_numpy(offsets_np).to(dev)
  proj = SphericalProjector(H, W, 3.0, -25.0).project(pts, offsets, want_image=False, want_idx=False,
                                                      want_point_outputs=True)
  cl = Clustering()

  # counts from the oracle, and its answer for a parity check of the timed output
  keys_np, px_np, py_np = proj["keys"].cpu().numpy(), proj["proj_x"].cpu().numpy(), proj["proj_y"].cpu().numpy()
  pts_np, lab_np = pts.cpu().numpy(), lab.cpu().numpy()
  nodes = tested = edges = 0
  want = np.zeros(total, np.int32)
  for b in range(B):
    sl = slice(offsets_np[b], offsets_np[b + 1])
    want[sl], _, st = PI.scan_instances(pts_np[sl], keys_np[b], px_np[sl], py_np[sl], lab_np[sl], KITTI_THINGS,
                                        cl.rows, cl.cols, cl.wrap, cl.tau, cl.min_points)
    nodes, tested, edges = nodes + st["nodes"], tested + st["edges_tested"], edges + st["edges"]
  nbytes = 40 * B * H * W + 52 * nodes + 44 * total

  lib = _lib.load()
  scratch = torch.empty(lib.pcls_point_instances_scratch_bytes(B, H, W) // 4, dtype=torch.float32, device=dev)
  inst = torch.empty(total, dtype=torch.int32, device=dev)
  counts = torch.empty(B, dtype=torch.int32, device=dev)
  s = torch.cuda.current_stream().cuda_stream
  args = (pts.data_ptr(), proj["keys"].data_ptr(), offsets.data_ptr(), B, H, W, total, proj["proj_x"].data_ptr(),
          proj["proj_y"].data_ptr(), lab.data_ptr(), 20, KITTI_THINGS, cl.rows, cl.cols, int(cl.wrap), cl.tau,
          cl.min_points, scratch.data_ptr(), inst.data_ptr(), counts.data_ptr(), s)
  _lib.check(lib.pcls_point_instances(*args), "pcls_point_instances")
  torch.cuda.synchronize()
  parity = bool(np.array_equal(inst.cpu().numpy(), want))
  kern_ms = []
  for _ in range(a.reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.kernel_calls):
      lib.pcls_point_instances(*args)
    e1.record()
    _lib.check(lib.pcls_point_instances(*args), "pcls_point_instances")
    torch.cuda.synchronize()
    kern_ms.append(e0.elapsed_time(e1) / a.kernel_calls)
  t = statistics.median(kern_ms)

  # per-kernel split (profiler run of its own)
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(10):
      lib.pcls_point_instances(*args)
    torch.cuda.synchronize()
  split = {}
  for ev in prof.key_averages():
    if "instances_" in ev.key:
      us = getattr(ev, "device_time_total", None)
      if us is None:
        us = ev.cuda_time_total
      name = ev.key.split("(")[0].replace("void ", "").replace("pcls::", "")
      split[name] = round(split.get(name, 0.0) + us / 10 / 1e3, 4)

  report = {"tool": "tools/point_instances_bench.py", "gpu": gpu_info(), "scans": B, "points": total, "H": H, "W": W,
            "clustering": {"tau": cl.tau, "rows": cl.rows, "cols": cl.cols, "min_points": cl.min_points,
                           "wrap": cl.wrap, "thing_mask": hex(KITTI_THINGS)},
            "nodes": nodes, "node_pairs_tested": tested, "edges": edges,
            "instances": int(counts.sum().item()), "parity_with_oracle": parity,
            "peak_hbm_GBps": peaks["hbm_gbs"], "peak_source": peaks["source"],
            "kernel": {"ms_median": round(t, 4), "ms_reps": kern_ms, "calls_per_rep": a.kernel_calls,
                       "algorithmic_bytes": nbytes, "GBps": nbytes / (t / 1e3) / 1e9,
                       "frac_of_hbm_peak": nbytes / (t / 1e3) / 1e9 / peaks["hbm_gbs"],
                       "per_kernel_ms": split}}
  print(json.dumps(report), flush=True)

  mc = config_map["squeezesegv2kitti"]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(1)
  seg = ScanSegmenter(model, 3.0, -25.0)
  knn = KNN()
  variants = {
    "knn": lambda: seg.segment_device(pts, offsets, want_point_labels=True, knn=knn),
    "knn_instances": lambda: seg.segment_device(pts, offsets, want_point_labels=True, knn=knn, instances=cl),
  }
  for step in variants.values():
    for _ in range(3):
      step()
  res = variants["knn_instances"]()
  torch.cuda.synchronize()
  ms = {k: [] for k in variants}
  for _ in range(a.reps):
    for name, step in variants.items():      # alternating: each repetition times every variant once
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for _ in range(a.steps):
        step()
      e1.record()
      torch.cuda.synchronize()
      ms[name].append(e0.elapsed_time(e1) / a.steps)
  med = {k: statistics.median(v) for k, v in ms.items()}
  report["step"] = {"network": "squeezesegv2", "config": "squeezesegv2kitti", "steps": a.steps, "reps": a.reps,
                    "ms_per_step": {k: round(v, 4) for k, v in med.items()}, "ms_per_step_reps": ms,
                    "spread_ms": {k: [min(v), max(v)] for k, v in ms.items()},
                    "scans_per_s": {k: B / (v / 1e3) for k, v in med.items()},
                    "overhead_of_instances": med["knn_instances"] / med["knn"] - 1.0,
                    "points_with_an_instance": int((res["instances"] > 0).sum().item()),
                    "instances_per_batch": int(res["instance_counts"].sum().item())}
  print(json.dumps(report["step"]), flush=True)
  model._release()
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump(report, f, indent=1)


if __name__ == "__main__":
  main()
