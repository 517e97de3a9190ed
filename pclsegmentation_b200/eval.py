"""Evaluation CLI - same flags and report as pcl_segmentation/eval.py (:33-82): per-class IoU / recall / precision and
the mean IoU over ``<data_path>/<image_set>/*.npy``.

    python -m pclsegmentation_b200.eval -d ./dataset -i val -m squeezesegv2 -n squeezesegv2 -p weights.npz
    torchrun --nproc-per-node 8 -m pclsegmentation_b200.eval ...      # frames sharded over 8 GPUs, one NCCL all-reduce

The TFRecord round trip of the reference (data_loader.py:252-330) is an I/O detour with no arithmetic of its own and
is skipped: the ``.npy`` frames go straight to the GPU, where the input stage, forward, head and the confusion-matrix
update run; only the final [NC,NC] matrix returns to the host.
"""
import argparse
import glob
import os

import numpy as np

from .inference import load_model_weights
from .pipeline import Evaluator, shard_files
from .tta import add_tta_flags, from_args
from .utils.args_loader import load_model_config


def evaluation(arg):
  import torch
  import torch.distributed as dist
  from .sharding import Communicator, env_rank
  rank, local_rank, world = env_rank()
  torch.cuda.set_device(local_rank)
  comm = None
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    comm = Communicator()

  config, model = load_model_config(arg.model, arg.config)
  config.DATA_AUGMENTATION = False
  load_model_weights(model, arg, verbose=rank == 0)

  files = shard_files(glob.glob(os.path.join(arg.data_path, arg.image_set, "*.npy")), comm)
  ev = Evaluator(model, comm, tta=from_args(arg.tta, arg.tta_shifts))
  if rank == 0:
    print("Performing Evaluation")
  for i in range(0, len(files), arg.batch):
    samples = np.stack([np.load(f) for f in files[i:i + arg.batch]])   # float64 files are narrowed on the device
    ev.update(samples)
  rep = ev.finish()

  if rank == 0:
    for i, cls in enumerate(config.CLASSES):
      print(cls.upper())
      print("IoU:       " + str(rep["iou"][i]))
      print("Recall:    " + str(rep["recall"][i]))
      print("Precision: " + str(rep["precision"][i]))
      print("")
    print("MIoU: {} ".format(rep["miou"]))
  if world > 1:
    comm.close()
    dist.destroy_process_group()
  return rep


def main(argv=None):
  parser = argparse.ArgumentParser(description='Parse Flags for the evaluation script!')
  parser.add_argument('-d', '--data_path', type=str, help='Absolute path to the dataset')
  parser.add_argument('-i', '--image_set', type=str, default="val", help='Default: `val`. But can also be train, val or test')
  parser.add_argument('-t', '--eval_dir', type=str, help="Kept for CLI compatibility (the reference writes nothing there)")
  parser.add_argument('-p', '--path_to_model', type=str, help='Path to the model: Keras SavedModel dir / checkpoint prefix (read without TensorFlow) or .npz')
  parser.add_argument('-m', '--model', type=str, help='Model name either `squeezesegv2`, `darknet53`, `darknet21`')
  parser.add_argument('-n', '--config', type=str, default='squeezesegv2',
                      help='Which configuration `squeezesegv2`, `squeezesegv2kitti`, `squeezesegv2nuscenes`, '
                           '`darknet53`, `darknet21`, `darknet53kitti`')
  parser.add_argument('-b', '--batch', type=int, default=8, help='frames per forward call (the reference uses 1)')
  parser.add_argument('--random_init', action='store_true', help='run without --path_to_model on Keras-default weights')
  add_tta_flags(parser)
  return evaluation(parser.parse_args(argv))


if __name__ == '__main__':
  main()
