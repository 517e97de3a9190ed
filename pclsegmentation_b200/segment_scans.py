"""Raw scans -> one label per point: projection, forward and per-point labels on the GPU, written as SemanticKITTI
``.label`` files (uint32, one word per point), optionally scored point-wise against label files.

    python -m pclsegmentation_b200.segment_scans --scans 'seq/08/velodyne/*.bin' -m darknet53 -n darknet53kitti \\
        -p weights.npz --learning_map semantic-kitti.yaml --output_dir out/08/predictions \\
        [--labels 'seq/08/labels/*.label']

Per point the label comes from the k-NN vote over the range image (``pipeline.KNN()`` defaults, the post-processing
published with RangeNet++) or, with --no_knn, from the point's own pixel.  With --learning_map the class ids are mapped
back through the yaml's ``learning_map_inv`` (what a SemanticKITTI submission needs) and the ground truth through its
``learning_map``; without it the class ids are written and the ground truth is taken as raw ids.  With --labels the
point-wise IoU / recall / precision / mIoU report is printed in eval.py's format.
"""
import argparse
import glob
import os

import numpy as np


def segment_scans(arg):
  from .dataset_convert import KITTI, ScanBatchLoader, learning_map_lut
  from .inference import load_model_weights
  from .pipeline import KNN, ScanEvaluator
  from .utils.args_loader import load_model_config

  config, model = load_model_config(arg.model or "squeezesegv2", arg.config)
  load_model_weights(model, arg)
  kitti = arg.format == KITTI
  fov_up, fov_down = (3.0, -25.0) if kitti else (12.0, -30.0)       # dataset_convert.main's defaults
  scans = sorted(glob.glob(arg.scans))
  labels = sorted(glob.glob(arg.labels)) if arg.labels else None
  if labels is not None and len(labels) != len(scans):
    raise SystemExit("%d scans but %d label files" % (len(scans), len(labels)))
  lut = inv = None
  if arg.learning_map:
    import yaml
    with open(arg.learning_map) as f:
      ym = yaml.safe_load(f)
    lut = learning_map_lut(ym["learning_map"])
    inv = learning_map_lut(ym["learning_map_inv"]).astype(np.uint32)
  ev = ScanEvaluator(model, fov_up, fov_down, label_lut=lut, knn=None if arg.no_knn else KNN())
  os.makedirs(arg.output_dir, exist_ok=True)
  loader = ScanBatchLoader(arg.format)
  for i in range(0, len(scans), arg.batch):
    files = scans[i:i + arg.batch]
    data = loader.load(files, labels[i:i + arg.batch] if labels is not None else None)
    if labels is not None:
      res = ev.update(data)
    else:
      res = ev.seg.segment_device(data["points"], data["offsets"], want_point_labels=True, knn=ev.knn)
    for f, lab in zip(files, ev.seg.point_labels(res, data["sizes"])):
      words = inv[lab] if inv is not None else lab.astype(np.uint32)
      words.astype(np.uint32).tofile(os.path.join(arg.output_dir, os.path.splitext(os.path.basename(f))[0] + ".label"))
  print("labelled %d scans -> %s" % (len(scans), arg.output_dir))
  if labels is None:
    return None
  rep = ev.finish()
  for c, cls in enumerate(config.CLASSES):
    print(cls.upper())
    print("IoU:       " + str(rep["iou"][c]))
    print("Recall:    " + str(rep["recall"][c]))
    print("Precision: " + str(rep["precision"][c]))
    print("")
  print("MIoU: {} ".format(rep["miou"]))
  if rep["dropped"]:
    print("WARNING: %d of %d points have a ground-truth id that is not a class id (0 .. %d) and are not scored%s"
          % (rep["dropped"], int(rep["confusion_matrix"].sum()) + rep["dropped"], config.NUM_CLASS - 1,
             "" if arg.learning_map else "; pass --learning_map to map raw label ids to classes"))
  return rep


def main(argv=None):
  ap = argparse.ArgumentParser(description="raw scans -> per-point labels (.label files), batched on the GPU")
  ap.add_argument("--scans", required=True, help="glob of .bin scan files")
  ap.add_argument("--format", choices=["kitti", "nuscenes"], default="kitti")
  ap.add_argument("-m", "--model", type=str, help="Model name either `squeezesegv2`, `darknet53`, `darknet21`")
  ap.add_argument("-n", "--config", type=str, default="squeezesegv2kitti", help="Which `mc` configuration to use")
  ap.add_argument("-p", "--path_to_model", type=str, help="SavedModel dir / checkpoint prefix / .npz")
  ap.add_argument("--random_init", action="store_true", help="run without --path_to_model on Keras-default weights")
  ap.add_argument("--batch", type=int, default=16, help="scans per forward call")
  ap.add_argument("--output_dir", required=True)
  ap.add_argument("--no_knn", action="store_true", help="each point takes its own pixel's label (no k-NN vote)")
  ap.add_argument("--labels", default=None, help="glob of .label (KITTI) / lidarseg .bin (nuScenes) files, same order: "
                                                 "print the point-wise report")
  ap.add_argument("--learning_map", default=None, help="yaml with `learning_map` / `learning_map_inv` (semantic-kitti.yaml)")
  return segment_scans(ap.parse_args(argv))


if __name__ == "__main__":
  main()
