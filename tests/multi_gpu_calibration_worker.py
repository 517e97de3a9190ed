"""torchrun worker for tests/test_gpu_calibration.py: every rank evaluates its contiguous shard of a synthetic val split
with a temperature fit (SqueezeSegV2, nuScenes config), the reliability and NLL sums are all-reduced, and rank 0 checks
them against what it computes alone over all frames: counts exactly, float64 sums within reordering, the same T*."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pclsegmentation_b200.calibration import Calibration  # noqa: E402
from pclsegmentation_b200.pipeline import Evaluator  # noqa: E402
from pclsegmentation_b200.sharding import Communicator, env_rank, shard_range  # noqa: E402
from pclsegmentation_b200.utils.args_loader import config_map, model_map  # noqa: E402
from tests.util import synth_range_images  # noqa: E402


def main():
  rank, local_rank, world = env_rank()
  torch.cuda.set_device(local_rank)
  dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
  comm = Communicator()
  mc = config_map["squeezesegv2nuscenes"]()
  mc.AZIMUTH_LEVEL = 256
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(1)
  n_frames = 13                               # ragged shards
  frames = synth_range_images(np.random.default_rng(78), n_frames, 32, 256, valid_rate=0.6, num_classes=11)
  lo, hi = shard_range(n_frames, rank, world)
  cal = Calibration(temperature=1.3, fit=True)
  ev = Evaluator(model, comm, calibration=cal)
  for i in range(lo, hi, 4):
    ev.update(frames[i:min(i + 4, hi)])
  got = ev.finish()["calibration"]
  ok = True
  if rank == 0:
    solo = Evaluator(model, None, calibration=cal)
    solo.update(frames)
    ref = solo.finish()["calibration"]
    r, w = got["reliability"], ref["reliability"]
    ok = bool(np.array_equal(r["bin_count"], w["bin_count"]) and r["count"] == w["count"] > 0 and
              np.allclose(r["bin_confidence"], w["bin_confidence"], rtol=1e-12, atol=0) and
              np.array_equal(r["bin_accuracy"], w["bin_accuracy"]) and got["nll"]["counted"] == ref["nll"]["counted"] and
              np.allclose(got["nll"]["nll"], ref["nll"]["nll"], rtol=1e-12, atol=0) and
              abs(got["nll"]["t_star"] / ref["nll"]["t_star"] - 1) < 1e-9)
    print(json.dumps({"ok": ok, "world": world, "pixels": int(r["count"]), "t_star": got["nll"]["t_star"]}))
  # every rank must hold the same T*
  t = torch.tensor([got["nll"]["t_star"]], dtype=torch.float64, device="cuda")
  t0 = t.clone()
  dist.broadcast(t0, src=0)
  same = bool(torch.equal(t, t0))
  comm.close()
  dist.destroy_process_group()
  sys.exit(0 if (ok and same) else 1)


if __name__ == "__main__":
  main()
