"""torchrun worker for tests/test_gpu_dataset_stats.py: every rank reduces its contiguous shard of a seeded frame set with
DatasetStats, finish() gathers the per-frame rows over torch.distributed, and rank 0 checks the result bit for bit
against the statistics it computes alone over all frames."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pclsegmentation_b200.dataset_stats import DatasetStats  # noqa: E402
from pclsegmentation_b200.sharding import Communicator, env_rank, shard_range  # noqa: E402
from pclsegmentation_b200.utils.args_loader import config_map  # noqa: E402
from tests.util import synth_range_images  # noqa: E402


def main():
  rank, local_rank, world = env_rank()
  torch.cuda.set_device(local_rank)
  dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
  comm = Communicator()
  mc = config_map["squeezesegv2kitti"]()
  n_frames, H, W = 13, 64, 512                              # ragged shards
  frames = synth_range_images(np.random.default_rng(78), n_frames, H, W, valid_rate=0.6).astype(np.float64)
  lo, hi = shard_range(n_frames, rank, world)
  st = DatasetStats(mc, H, W)
  for i in range(lo, hi, 4):
    st.update(frames[i:min(i + 4, hi)])
  rep = st.finish(comm)
  as_bytes = lambda r: {k: (v.tobytes() if isinstance(v, np.ndarray) else v) for k, v in r.items()}
  got = as_bytes(rep)
  ok = True
  if rank == 0:
    solo = DatasetStats(mc, H, W)
    solo.update(frames)
    ok = got == as_bytes(solo.finish()) and rep["frames"] == n_frames
    print(json.dumps({"ok": ok, "world": world, "valid": rep["valid"], "mean": rep["mean"].reshape(-1).tolist()}))
  # every rank holds the same result
  everyone = [None] * world
  dist.all_gather_object(everyone, got)
  same = all(e == got for e in everyone)
  comm.close()
  dist.destroy_process_group()
  sys.exit(0 if (ok and same) else 1)


if __name__ == "__main__":
  main()
