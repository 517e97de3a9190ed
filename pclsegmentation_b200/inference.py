"""Inference CLI - same flags and outputs as pcl_segmentation/inference.py (:36-132): for every ``*.npy`` sample
matched by --input_path it writes ``pred_<name>.npy`` (int32 [H,W] class ids) plus the colour-mapped PNGs.

    python -m pclsegmentation_b200.inference -d './samples/*.npy' -m squeezesegv2 -t ./out -p weights.npz

Differences, all documented in DESIGN.md: --path_to_model takes the reference's SavedModel directory / checkpoint prefix
(its TensorBundle is read without TensorFlow, utils/tensor_bundle.py) or an ``.npz`` container keyed by Keras attribute
paths (a missing path is an error; --random_init runs an untrained, Keras-default-initialised network on purpose); --config selects the ``mc`` factory
(the reference hard-codes SqueezeSegV2Config, inference.py:37 - that is the default here); the normalise / mask stage
(inference.py:50-62) runs fused on the GPU; --batch frames go through the network per call.
"""
import argparse
import glob
import os

import numpy as np
import torch

from .calibration import add_temperature_flag, confidence, raw_mask
from .device import samples_to_device
from .mc_dropout import add_mc_flags, check_exclusive, forward_mc, from_args as mc_from_args
from .tta import add_tta_flags, forward_tta, from_args
from .utils.args_loader import load_model_config
from .utils.util import normalize


def load_model_weights(model, arg, verbose=True):
  """--path_to_model given: ALWAYS load it (a SavedModel directory, a checkpoint PREFIX - which never exists as a file,
  only `<prefix>.index` / `.data-*` do - or an .npz); a wrong path raises FileNotFoundError like the reference's
  `tf.keras.models.load_model` (inference.py:39).  Random (Keras-default) weights only on the explicit --random_init."""
  if arg.path_to_model:
    if not str(arg.path_to_model).endswith(".npz") or os.path.exists(arg.path_to_model):
      model.load_weights(arg.path_to_model)    # tensor_bundle.resolve_prefix raises FileNotFoundError for a bad path
    else:
      raise FileNotFoundError("--path_to_model %r does not exist" % arg.path_to_model)
  elif getattr(arg, "random_init", False):
    if verbose:
      print("--random_init: using the Keras-default initialisation (untrained network)")
  else:
    raise SystemExit("--path_to_model is required (SavedModel dir / checkpoint prefix / .npz); pass --random_init to run "
                     "an untrained network on purpose")


def inference(arg):
  import torch
  config, model = load_model_config(arg.model or "squeezesegv2", arg.config)
  load_model_weights(model, arg)

  if not os.path.exists(arg.output_dir):
    os.makedirs(arg.output_dir)
  none = config.CLASSES.index("None")
  tta = from_args(arg.tta, arg.tta_shifts)
  if arg.confidence and tta is not None and arg.temperature != 1.0:
    raise SystemExit("--tta merges probabilities, not logits: --confidence with --tta needs --temperature 1")
  mcd = mc_from_args(arg)
  if mcd is not None:
    if arg.confidence and arg.temperature != 1.0:
      raise SystemExit("MC dropout cannot be combined with a softmax temperature: --confidence needs --temperature 1")
    try:
      check_exclusive(mcd, tta)
    except ValueError as e:
      raise SystemExit(str(e))
  files = sorted(glob.iglob(arg.input_path))
  for i in range(0, len(files), arg.batch):
    chunk = files[i:i + arg.batch]
    samples = np.stack([np.load(f) for f in chunk])          # float64 on disk: uploaded as is, narrowed on the device
    x = samples_to_device(samples)
    unc = None
    if mcd is not None:
      res = forward_mc(model, x, mcd)
      unc = torch.stack([res["entropy"], res["mutual_information"]], dim=-1).cpu().numpy()   # [B,H,W,2]: H, MI
    elif tta is not None:
      res = forward_tta(model, x, tta, want_probabilities=arg.confidence)
    else:
      res = model.forward_device(x, None, mean=config.INPUT_MEAN, std=config.INPUT_STD, want_probabilities=False,
                                 want_logits=arg.confidence)
    conf = None
    if arg.confidence and mcd is not None:
      conf = res["confidence"].cpu().numpy()
    elif arg.confidence:
      src = dict(probs=res["probabilities"]) if tta is not None else dict(logits=res["logits"])
      conf = confidence(config.NUM_CLASS, mask=raw_mask(x, config), temperature=arg.temperature,
                        **src)["confidence"].cpu().numpy()
    predictions = res["predictions"].cpu().numpy()
    for k, (f, sample, pred) in enumerate(zip(chunk, samples, predictions)):
      print("Process: {0}".format(f))
      file_name = os.path.splitext(os.path.basename(f))[0]
      np.save(os.path.join(arg.output_dir, 'pred_' + file_name + '.npy'), pred)
      if conf is not None:
        np.save(os.path.join(arg.output_dir, 'conf_' + file_name + '.npy'), conf[k])
      if unc is not None:
        np.save(os.path.join(arg.output_dir, 'unc_' + file_name + '.npy'), unc[k])
      if arg.no_plots:
        continue
      from PIL import Image
      mask = sample[:, :, 4] > 0
      label = sample[:, :, 5].copy()
      label[~mask] = none
      intensity = np.where(mask, (sample[:, :, 3] - config.INPUT_MEAN[0, 0, 3]) / config.INPUT_STD[0, 0, 3], 0.0)
      depth_map = Image.fromarray((255 * normalize(intensity)).astype(np.uint8))
      for tag, lab in (('plot_', pred), ('plot_gt_', label.astype(np.int32))):
        label_map = Image.fromarray((255 * config.CLS_COLOR_MAP[lab]).astype(np.uint8))
        blend_map = Image.blend(depth_map.convert('RGBA'), label_map.convert('RGBA'), alpha=1.0)
        blend_map.save(os.path.join(arg.output_dir, tag + file_name + '.png'))


def main(argv=None):
  parser = argparse.ArgumentParser(description='Parse Flags for the inference script!')
  parser.add_argument('-d', '--input_path', type=str,
                      help='Input LiDAR scans to be detected. Must be a glob pattern input such as'
                           '`./data/samples/*.npy` !')
  parser.add_argument('-m', '--model', type=str, help='Model name either `squeezesegv2`, `darknet53`, `darknet21`')
  parser.add_argument('-t', '--output_dir', type=str,
                      help="Directory where to write the model predictions and visualizations")
  parser.add_argument('-p', '--path_to_model', type=str, help='Path to the model: Keras SavedModel dir / checkpoint prefix (read without TensorFlow) or .npz')
  parser.add_argument('-n', '--config', type=str, default='squeezesegv2', help='Which `mc` configuration to use')
  parser.add_argument('-b', '--batch', type=int, default=8, help='frames per forward call')
  parser.add_argument('--no_plots', action='store_true', help='only write pred_*.npy')
  parser.add_argument('--random_init', action='store_true', help='run without --path_to_model on Keras-default weights')
  add_tta_flags(parser)
  add_mc_flags(parser)
  parser.add_argument('--confidence', action='store_true',
                      help='also write conf_<name>.npy: float32 [H,W] max softmax(logits / T) per pixel, 0 at empty pixels')
  add_temperature_flag(parser)
  inference(parser.parse_args(argv))


if __name__ == '__main__':
  main()
