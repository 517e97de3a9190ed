#!/usr/bin/env python
"""Cost of pcls_dataset_stats: the kernel alone on batches of 64 frames of 64 x 2048 resident in HBM (float64 x 6
channels = 403 MB per batch, more than the 126 MB of L2; two batches alternated so that no call re-reads what the last
one left in L2), CUDA events over --calls launches after a warm-up.  Algorithmic bytes = the frames read once
(B*H*W*C*sizeof); the HBM peak is bench.py's.  Also the float32 / 5-channel variant, and the CLI end to end on .npy
files (np.load + upload + kernel): a host- and disk-bound number, not the kernel's.

    python tools/dataset_stats_bench.py [--calls 50] [--out profiles/dataset_stats_bench_b200.json]
"""
import argparse
import ctypes
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--calls", type=int, default=50)
  ap.add_argument("--cli-frames", type=int, default=128)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("dataset_stats_bench: no CUDA device (there is no CPU fallback)")
  from bench import measured_peaks
  from pclsegmentation_b200 import _lib, dataset_stats
  from tools.point_labels_bench import gpu_info
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  peaks = measured_peaks()
  lib = _lib.load()
  B, H, W, NC = 64, 64, 2048, 20
  shift = np.array([-0.047, 0.365, -0.855, 0.2198, 8.3568])
  sh = shift.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
  report = {"tool": "tools/dataset_stats_bench.py", "gpu": gpu_info(), "B": B, "H": H, "W": W, "calls": a.calls,
            "peak_hbm_GBps": peaks["hbm_gbs"], "peak_source": peaks["source"], "kernel": []}
  for dtype, C in ((torch.float64, 6), (torch.float64, 5), (torch.float32, 6), (torch.float32, 5)):
    bufs = []
    for seed in range(2):
      g = torch.Generator(device=dev).manual_seed(seed)
      x = torch.rand((B, H, W, C), dtype=dtype, device=dev, generator=g) * 40.0
      x[..., 4] -= 8.0                                                # ~20 % invalid pixels
      if C == 6:
        x[..., 5] = torch.floor(x[..., 5] * 0.55)                    # labels 0 .. 21: some dropped
      bufs.append(x)
    sums = torch.empty((B, 5, 4), dtype=torch.float64, device=dev)
    valid = torch.empty(B, dtype=torch.int64, device=dev)
    cnt = [torch.zeros(n, dtype=torch.int64, device=dev) for n in (H, W, NC, 1)]
    s = torch.cuda.current_stream().cuda_stream

    def call(i):
      return lib.pcls_dataset_stats(bufs[i % 2].data_ptr(), 1 if dtype == torch.float64 else 0, C, B, H, W, sh, NC,
                                    sums.data_ptr(), valid.data_ptr(), cnt[0].data_ptr(), cnt[1].data_ptr(),
                                    cnt[2].data_ptr() if C == 6 else None, cnt[3].data_ptr() if C == 6 else None, s)
    for i in range(4):
      _lib.check(call(i), "pcls_dataset_stats")
    torch.cuda.synchronize()
    times = []
    for rep in range(3):
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      for i in range(a.calls):
        call(i)
      e1.record()
      torch.cuda.synchronize()
      times.append(e0.elapsed_time(e1) / a.calls)
    _lib.check(call(0), "pcls_dataset_stats")
    torch.cuda.synchronize()
    by = B * H * W * C * bufs[0].element_size()
    ms = sorted(times)[1]
    entry = {"dtype": str(dtype).replace("torch.", ""), "channels": C, "algorithmic_bytes": by, "ms_reps": times,
             "ms": ms, "GBps": by / (ms / 1e3) / 1e9, "frac_of_hbm_peak": by / (ms / 1e3) / 1e9 / peaks["hbm_gbs"],
             "frames_per_s": B / (ms / 1e3)}
    report["kernel"].append(entry)
    print(json.dumps(entry), flush=True)
    del bufs, x
    torch.cuda.empty_cache()

  # CLI end to end on float64 .npy files (the converter's output format): host- and disk-bound
  with tempfile.TemporaryDirectory() as d:
    rng = np.random.default_rng(0)
    one = rng.uniform(0, 40, (H, W, 6))
    for i in range(a.cli_frames):
      np.save(os.path.join(d, "%d.npy" % i), one)
    dataset_stats.main(["-d", os.path.join(d, "*.npy"), "-b", "64"])       # warm-up (and page cache)
    t0 = time.perf_counter()
    rep = dataset_stats.main(["-d", os.path.join(d, "*.npy"), "-b", "64"])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    report["cli_npy_end_to_end"] = {
        "what": "python -m pclsegmentation_b200.dataset_stats -d '*.npy' -b 64 on %d float64 64x2048x6 files just "
                "written (page cache warm): np.load + stack + upload + kernel + report; host- and disk-bound" % a.cli_frames,
        "frames": rep["frames"], "s": dt, "frames_per_s": rep["frames"] / dt}
  print(json.dumps(report))
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump(report, f, indent=1)


if __name__ == "__main__":
  main()
