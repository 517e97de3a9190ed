"""Evaluation CLI - same flags and report as pcl_segmentation/eval.py (:33-82): per-class IoU / recall / precision and
the mean IoU over ``<data_path>/<image_set>/*.npy``.

    python -m pclsegmentation_b200.eval -d ./dataset -i val -m squeezesegv2 -n squeezesegv2 -p weights.npz
    torchrun --nproc-per-node 8 -m pclsegmentation_b200.eval ...      # frames sharded over 8 GPUs, one NCCL all-reduce

The TFRecord round trip of the reference (data_loader.py:252-330) is an I/O detour with no arithmetic of its own and
is skipped: the ``.npy`` frames go straight to the GPU, where the input stage, forward, head and the confusion-matrix
update run; only the final [NC,NC] matrix returns to the host.

--calibration prints the reliability of the confidences at --temperature (ECE, MCE, accuracy, mean confidence and a
per-bin table) after the mIoU report.  --fit_temperature also accumulates the NLL on a log-spaced temperature grid,
prints NLL(1), the fitted T* and NLL(T*), and runs a second pass over the same frames for the reliability at T*.
--calibration_json FILE writes these reports.  Under torchrun the sums are all-reduced, so every rank fits the same T*.
"""
import argparse
import glob
import json
import os

import numpy as np

from .inference import load_model_weights
from .calibration import Calibration, add_temperature_flag
from .mc_dropout import add_mc_flags, from_args as mc_from_args
from .pipeline import Evaluator, shard_files
from .tta import add_tta_flags, from_args
from .utils.args_loader import load_model_config


def evaluation(arg):
  import torch
  import torch.distributed as dist
  from .sharding import Communicator, env_rank, shard_range
  rank, local_rank, world = env_rank()
  torch.cuda.set_device(local_rank)
  comm = None
  if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    comm = Communicator()

  config, model = load_model_config(arg.model, arg.config)
  config.DATA_AUGMENTATION = False
  load_model_weights(model, arg, verbose=rank == 0)

  all_files = glob.glob(os.path.join(arg.data_path, arg.image_set, "*.npy"))
  files = shard_files(all_files, comm)
  tta = from_args(arg.tta, arg.tta_shifts)
  mcd = mc_from_args(arg)
  if mcd is not None and comm is not None:
    # the rank's first frame keeps its single-GPU global id: the same masks, so the same integer histograms
    mcd.next_frame = shard_range(len(all_files), comm.rank, comm.world_size)[0]
  cal = None
  if arg.calibration or arg.fit_temperature or arg.calibration_json:
    cal = Calibration(temperature=arg.temperature, n_bins=arg.bins, fit=arg.fit_temperature)
  try:
    ev = Evaluator(model, comm, tta=tta, calibration=cal, mc_dropout=mcd)
  except ValueError as e:
    raise SystemExit(str(e))
  if rank == 0:
    print("Performing Evaluation")

  def run(evaluator):
    for i in range(0, len(files), arg.batch):
      samples = np.stack([np.load(f) for f in files[i:i + arg.batch]])   # float64 files are narrowed on the device
      evaluator.update(samples)
    return evaluator.finish()

  rep = run(ev)

  if rank == 0:
    for i, cls in enumerate(config.CLASSES):
      print(cls.upper())
      print("IoU:       " + str(rep["iou"][i]))
      print("Recall:    " + str(rep["recall"][i]))
      print("Precision: " + str(rep["precision"][i]))
      print("")
    print("MIoU: {} ".format(rep["miou"]))
    if mcd is not None:
      print_mc_report(rep["mc_dropout"], "pixels")
  if cal is not None:
    calib = rep["calibration"]
    if rank == 0:
      print_reliability(calib["reliability"], cal.temperature, "pixels")
    fit = calib["nll"]
    if cal.fit and fit["t_star"] is None:
      if rank == 0:
        print("no temperature fit: no pixel has a class label")
    elif cal.fit:
      again = Calibration(temperature=fit["t_star"], n_bins=cal.n_bins)
      calib["fitted"] = run(Evaluator(model, comm, tta=tta, calibration=again))["calibration"]
      if rank == 0:
        print("TEMPERATURE FIT (%d pixels, %d temperatures in [%g, %g])" % (fit["counted"], len(fit["temperatures"]),
                                                                           cal.grid[0], cal.grid[1]))
        print("NLL(1):    %.6f" % fit["nll_at_1"])
        print("T*:        %.6f" % fit["t_star"])
        print("NLL(T*):   %.6f" % calib["fitted"]["nll"]["nll_at_temperature"])
        if fit["at_edge"]:
          print("WARNING: the NLL is smallest at the end of the grid; T* may lie outside [%g, %g]" % cal.grid[:2])
        print_reliability(calib["fitted"]["reliability"], fit["t_star"], "pixels")
    if rank == 0 and arg.calibration_json:
      with open(arg.calibration_json, "w") as f:
        json.dump(_jsonable(calib), f, indent=1)
  if world > 1:
    comm.close()
    dist.destroy_process_group()
  return rep


def print_mc_report(m, what):
  """The MC-dropout report: T, rate, seed, the AUROC of H and MI for detecting errors, ECE / MCE of the mean."""
  u, r = m["uncertainty"], m["reliability"]
  print("MC DROPOUT T = %d, rate = %g, seed = %d (%d %s, %d errors)" % (m["passes"], m["rate"], m["seed"], u["count"],
                                                                        what, u["errors"]))
  print("AUROC(H):        %.6f" % u["auroc_entropy"])
  print("AUROC(MI):       %.6f" % u["auroc_mi"])
  print("ECE (mean conf): %.6f" % r["ece"])
  print("MCE (mean conf): %.6f" % r["mce"])


def print_reliability(r, temperature, what):
  """The reliability report of ``metrics.Reliability.result()``."""
  print("RELIABILITY at T = %g (%d %s, %d bins)" % (temperature, r["count"], what, len(r["bin_count"])))
  print("ECE:             %.6f" % r["ece"])
  print("MCE:             %.6f" % r["mce"])
  print("Accuracy:        %.6f" % r["accuracy"])
  print("Mean confidence: %.6f" % r["mean_confidence"])
  print("bin              count    accuracy  confidence")
  for lo, hi, n, acc, conf in zip(r["bin_lo"], r["bin_hi"], r["bin_count"], r["bin_accuracy"], r["bin_confidence"]):
    print("[%.3f, %.3f) %10d  %10.6f  %10.6f" % (lo, hi, n, acc, conf))


def _jsonable(v):
  if isinstance(v, dict):
    return {k: _jsonable(x) for k, x in v.items()}
  if isinstance(v, (list, tuple)):
    return [_jsonable(x) for x in v]
  if isinstance(v, np.ndarray):
    return _jsonable(v.tolist())
  if isinstance(v, np.generic):
    return v.item()
  if isinstance(v, float) and not np.isfinite(v):
    return None
  return v


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
  add_mc_flags(parser)
  parser.add_argument('--calibration', action='store_true',
                      help='print the reliability of the confidences (ECE, MCE, per-bin table) at --temperature')
  parser.add_argument('--fit_temperature', action='store_true',
                      help='also fit the softmax temperature T* on the NLL and report the reliability at T*')
  parser.add_argument('--calibration_json', type=str, default=None, help='write the calibration report to this file')
  parser.add_argument('--bins', type=int, default=15, help='reliability bins (1..64)')
  add_temperature_flag(parser)
  return evaluation(parser.parse_args(argv))


if __name__ == '__main__':
  main()
