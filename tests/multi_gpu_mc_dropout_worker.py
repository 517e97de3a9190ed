"""torchrun worker for tests/test_gpu_mc_dropout.py: every rank evaluates its contiguous shard of a synthetic val split
with MC dropout (SqueezeSegV2, nuScenes config), starting its frame counter at the shard's first global frame index as
the eval CLI does; the confusion matrix and the uncertainty / reliability bins are all-reduced, and rank 0 checks them
against what it computes alone over all frames: the matrix and every integer bin exactly."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pclsegmentation_b200.mc_dropout import MCDropout  # noqa: E402
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
  frames = synth_range_images(np.random.default_rng(79), n_frames, 32, 256, valid_rate=0.6, num_classes=11)
  lo, hi = shard_range(n_frames, rank, world)
  mcd = MCDropout(passes=3, seed=17, rate=0.4)
  mcd.next_frame = lo
  ev = Evaluator(model, comm, mc_dropout=mcd)
  for i in range(lo, hi, 4):
    ev.update(frames[i:min(i + 4, hi)])
  got = ev.finish()
  ok = True
  if rank == 0:
    solo = Evaluator(model, None, mc_dropout=MCDropout(passes=3, seed=17, rate=0.4))
    for i in range(0, n_frames, 5):           # another batching: the masks follow the global frame ids
      solo.update(frames[i:i + 5])
    ref = solo.finish()
    g, r = got["mc_dropout"], ref["mc_dropout"]
    ok = bool(np.array_equal(got["confusion_matrix"], ref["confusion_matrix"]) and
              all(np.array_equal(g["uncertainty"][k], r["uncertainty"][k])
                  for k in ("entropy_count", "entropy_correct", "mi_count", "mi_correct")) and
              np.array_equal(g["reliability"]["bin_count"], r["reliability"]["bin_count"]) and
              np.array_equal(g["reliability"]["bin_accuracy"], r["reliability"]["bin_accuracy"]) and
              g["uncertainty"]["count"] > 0 and g["uncertainty"]["auroc_mi"] == r["uncertainty"]["auroc_mi"])
    print(json.dumps({"ok": ok, "world": world, "pixels": g["uncertainty"]["count"],
                      "auroc_mi": g["uncertainty"]["auroc_mi"]}))
  comm.close()
  dist.destroy_process_group()
  sys.exit(0 if ok else 1)


if __name__ == "__main__":
  main()
