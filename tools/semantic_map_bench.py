#!/usr/bin/env python
"""Cost of semantic map fusion: a synthetic KITTI-sized sequence of 256 scans of ~120 k points (tests.util.synth_scan,
16 distinct scans reused) along a ~2 km trajectory (7.8 m between scans, a gentle curve, a few degrees of roll and
pitch), in batches of 16 scans, random labels of 20 classes.  Every scan is new random points, so nearly every voting
point makes its own voxel: more voxels than a real static scene gives, the expensive side for the table.

  kernel   pcls_semantic_map_vote over the whole sequence into an empty, pre-sized table (inserts and counts), then
           pcls_semantic_map_query over the whole sequence; CUDA events around the 16 calls, --reps repetitions, as
           points/s.
  table    voxels, final capacity under SemanticMap's growth rule (from 2^20 slots) and table bytes at 0.1 and 0.2 m.
  step     SqueezeSegV2-KITTI 64 x 2048 (random init + randomised BN) ScanSegmenter.segment_device with the k-NN vote
           over a 16-scan batch, without and with SemanticMap.vote of its point labels, alternating, --steps timed
           steps per repetition.
  parity   the export of the first 32 scans at 0.2 m and the query of those scans against oracle/semantic_map.py.

    python tools/semantic_map_bench.py [--steps 10] [--reps 5] [--out profiles/semantic_map_bench_b200.json]
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SCANS, BATCH, NC = 256, 16, 20


def trajectory(rng):
  poses = np.tile(np.eye(4), (SCANS, 1, 1))
  heading = 0.0
  pos = np.zeros(3)
  for i in range(SCANS):
    heading += 0.004 * np.sin(i / 20.0)
    pos = pos + 7.8 * np.array([np.cos(heading), np.sin(heading), 0.0])
    roll, pitch = np.deg2rad(rng.uniform(-2, 2, 2))
    c, s = np.cos(heading), np.sin(heading)
    rz = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]])
    rx = np.array([[1, 0, 0], [0, np.cos(roll), -np.sin(roll)], [0, np.sin(roll), np.cos(roll)]])
    ry = np.array([[np.cos(pitch), 0, np.sin(pitch)], [0, 1, 0], [-np.sin(pitch), 0, np.cos(pitch)]])
    poses[i, :3, :3] = rz @ ry @ rx
    poses[i, :3, 3] = pos
  return poses


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--reps", type=int, default=5)
  ap.add_argument("--out", default=None, help="also write the JSON report here")
  a = ap.parse_args()
  import torch
  if not torch.cuda.is_available():
    raise SystemExit("semantic_map_bench: no CUDA device (there is no CPU fallback)")
  from oracle import semantic_map as SM
  from pclsegmentation_b200 import _lib
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  from pclsegmentation_b200.semantic_map import SemanticMap, _pose_rows
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  from tests.util import synth_scan
  from tools.point_labels_bench import gpu_info
  torch.cuda.set_device(0)
  dev = torch.device("cuda", 0)
  rng = np.random.default_rng(0)
  base = [synth_scan(rng, int(rng.integers(115000, 125000))) for _ in range(BATCH)]
  base_labels = [rng.integers(0, NC, s.shape[0]).astype(np.int32) for s in base]
  poses = trajectory(rng)
  sizes = [s.shape[0] for s in base]
  pts = torch.from_numpy(np.concatenate(base)).to(dev)
  lab = torch.from_numpy(np.concatenate(base_labels)).to(dev)
  offs = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).to(dev)
  rows = [_pose_rows(poses[lo:lo + BATCH], BATCH, dev) for lo in range(0, SCANS, BATCH)]
  per_batch, total = int(pts.shape[0]), int(pts.shape[0]) * (SCANS // BATCH)
  lib = _lib.load()
  s = torch.cuda.current_stream().cuda_stream
  report = {"tool": "tools/semantic_map_bench.py", "gpu": gpu_info(), "scans": SCANS, "batch": BATCH,
            "points": total, "points_per_batch": per_batch, "num_classes": NC,
            "trajectory_m": float(np.linalg.norm(np.diff(poses[:, :3, 3], axis=0), axis=1).sum())}

  # table size under the growth rule
  report["table"] = {}
  for vs in (0.1, 0.2):
    m = SemanticMap(NC, voxel_size=vs)
    for j in range(len(rows)):
      m.vote(pts, offs, poses[j * BATCH:(j + 1) * BATCH], lab)
    report["table"]["%g" % vs] = {"voxels": m.num_voxels, "capacity": m.capacity,
                                  "bytes": m.capacity * (8 + 4 * NC)}
    del m
  torch.cuda.empty_cache()

  # kernel times: vote into an empty pre-sized table, then query, over the whole sequence
  vs = 0.2
  cap = report["table"]["0.2"]["capacity"]
  keys = torch.empty(cap, dtype=torch.int64, device=dev)
  counts = torch.empty((cap, NC), dtype=torch.int32, device=dev)
  state = torch.empty(2, dtype=torch.int64, device=dev)
  out = torch.empty(per_batch, dtype=torch.int32, device=dev)

  def vote_all():
    for r in rows:
      _lib.check(lib.pcls_semantic_map_vote(pts.data_ptr(), offs.data_ptr(), BATCH, per_batch, r.data_ptr(), vs, 0.0,
                                            50.0, lab.data_ptr(), NC, -1, keys.data_ptr(), counts.data_ptr(), cap,
                                            state.data_ptr(), s), "pcls_semantic_map_vote")

  def query_all():
    for r in rows:
      _lib.check(lib.pcls_semantic_map_query(pts.data_ptr(), offs.data_ptr(), BATCH, per_batch, r.data_ptr(), vs,
                                             lab.data_ptr(), NC, 0, 1, keys.data_ptr(), counts.data_ptr(), cap,
                                             out.data_ptr(), s), "pcls_semantic_map_query")

  vote_ms, query_ms = [], []
  for rep in range(a.reps + 1):
    keys.fill_(-1)
    counts.zero_()
    state.zero_()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    vote_all()
    e[1].record()
    query_all()
    e[2].record()
    torch.cuda.synchronize()
    if rep:                     # repetition 0 warms up
      vote_ms.append(e[0].elapsed_time(e[1]))
      query_ms.append(e[1].elapsed_time(e[2]))
  st = state.cpu().tolist()
  report["kernel"] = {"voxel_size": vs, "capacity": cap, "occupied": st[0], "failed_inserts": st[1],
                      "vote_ms_sequence": vote_ms, "query_ms_sequence": query_ms,
                      "vote_points_per_s": total / (statistics.median(vote_ms) / 1e3),
                      "query_points_per_s": total / (statistics.median(query_ms) / 1e3),
                      "vote_ms_per_batch": statistics.median(vote_ms) / len(rows),
                      "query_ms_per_batch": statistics.median(query_ms) / len(rows)}
  print(json.dumps(report["kernel"]), flush=True)
  del keys, counts
  torch.cuda.empty_cache()

  # parity on the first 32 scans
  m = SemanticMap(NC, voxel_size=0.2)
  for j in range(2):
    m.vote(pts, offs, poses[j * BATCH:(j + 1) * BATCH], lab)
  pts_np, offs_np = np.concatenate(base), np.concatenate([[0], np.cumsum(sizes)])
  lab_np = np.concatenate(base_labels)
  ks, ls = [], []
  for j in range(2):
    k, l = SM.voters(pts_np, offs_np, poses[j * BATCH:(j + 1) * BATCH], 0.2, lab_np, NC, -1, 0.0, 50.0)
    ks.append(k)
    ls.append(l)
  tk, tc = SM.table(np.concatenate(ks), np.concatenate(ls), NC)
  want, got = SM.export(tk, tc, 0.2), m.export()
  ok = all(np.array_equal(got[k], want[k]) for k in ("voxels", "counts", "labels"))
  q = m.relabel(pts, offs, poses[:BATCH], lab).cpu().numpy()
  ok = ok and np.array_equal(q, SM.relabel(pts_np, offs_np, poses[:BATCH], 0.2, lab_np, tk, tc))
  report["parity_with_oracle"] = bool(ok)
  del m

  # step time without and with the vote
  mc = config_map["squeezesegv2kitti"]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = 64, 2048
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(1)
  seg = ScanSegmenter(model, 3.0, -25.0)
  knn = KNN()
  m = SemanticMap(mc.NUM_CLASS, voxel_size=0.2, ignore_class=mc.CLASSES.index("None"))
  j = [0]

  def with_vote():
    res = seg.segment_device(pts, offs, want_point_labels=True, knn=knn)
    b = j[0] % len(rows)
    j[0] += 1
    m.vote(pts, offs, poses[b * BATCH:(b + 1) * BATCH], res["point_labels"])

  variants = {"knn": lambda: seg.segment_device(pts, offs, want_point_labels=True, knn=knn), "knn_vote": with_vote}
  for step in variants.values():
    for _ in range(3):
      step()
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
  report["step"] = {"network": "squeezesegv2", "config": "squeezesegv2kitti", "H": 64, "W": 2048, "steps": a.steps,
                    "reps": a.reps, "ms_per_step": {k: round(v, 4) for k, v in med.items()}, "ms_per_step_reps": ms,
                    "spread_ms": {k: [min(v), max(v)] for k, v in ms.items()},
                    "overhead_of_vote": med["knn_vote"] / med["knn"] - 1.0, "map_voxels_after": m.num_voxels}
  print(json.dumps(report["step"]), flush=True)
  model._release()
  if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
      json.dump(report, f, indent=1)


if __name__ == "__main__":
  main()
