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

With --instances every thing-class point also gets an instance id (``pipeline.Clustering``: connected components in
the range image, tuned by --cluster_tau / --cluster_rows / --cluster_cols / --min_points / --no_wrap), written to the
upper 16 bits of its word as in SemanticKITTI's panoptic labels.  With --labels in KITTI format the panoptic quality
report (PQ / SQ / RQ per thing class) follows the mIoU report; nuScenes lidarseg files carry no instance ids, so there
it is skipped.

With --tta (the mirror image) and / or --tta_shifts (rolls by that many columns, e.g. 0,1024) the forward runs over
those views of each scan's range image and their averaged probabilities decide the pixel labels (``tta.TTA``).

With --confidence each point's confidence is written next to its ``.label`` file as ``<name>.conf`` (raw float32, one
per point): the probability at --temperature T that the point's own pixel gives the point's label (0 for a point the
projection dropped).  With --labels the point-wise reliability report (ECE, MCE, per-bin table) follows the other
reports.

With --map (KITTI layout; needs --poses and --calib) the sequence is fused through a semantic map
(``semantic_map.SemanticMap``): pass 1 segments every batch as above and votes its point labels into a voxel map
registered by the sequence's poses ("None" casts no vote); pass 2 relabels every scan from the map and writes the fused
labels.  The pose of a scan is the integer stem of its file name (``000123.bin`` -> line 123 of poses.txt), so a glob
over part of a sequence works.  --map_keep things (default) keeps the thing classes of ``pipeline.Clustering`` as the
network labelled them, since moving objects would otherwise take the static votes under them.  --map_out writes the
map (``SemanticMap.save``).  With --labels a second report, headed FUSED (semantic map), follows the per-scan one.
"""
import argparse
import glob
import os

import numpy as np


def segment_scans(arg):
  from .dataset_convert import KITTI, ScanBatchLoader, learning_map_lut
  if arg.map:
    if arg.instances or arg.confidence or arg.mc_dropout is not None:
      raise SystemExit("--map cannot be combined with --instances, --confidence or --mc_dropout")
    if arg.format != KITTI:
      raise SystemExit("--map reads SemanticKITTI poses.txt / calib.txt; there is no nuScenes poses reader (the Python "
                       "API, semantic_map.SemanticMap, takes any poses)")
    if not arg.poses or not arg.calib:
      raise SystemExit("--map needs --poses (poses.txt) and --calib (calib.txt) of the sequence")
    if arg.map_min_votes < 1:
      raise SystemExit("--map_min_votes must be >= 1")
  from .inference import load_model_weights
  from .calibration import Calibration
  from .metrics import MeanIoU
  from .pipeline import KNN, Clustering, ScanEvaluator
  from .semantic_map import SemanticMap, kitti_lidar_poses, scan_pose_index
  from .tta import from_args
  from .mc_dropout import from_args as mc_from_args
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
  clustering = None
  if arg.instances:
    clustering = Clustering(tau=arg.cluster_tau, rows=arg.cluster_rows, cols=arg.cluster_cols,
                            min_points=arg.min_points, wrap=not arg.no_wrap)
  tta = from_args(arg.tta, arg.tta_shifts)
  mcd = mc_from_args(arg)
  cal = Calibration(temperature=arg.temperature, n_bins=arg.bins) if arg.confidence else None
  try:
    ev = ScanEvaluator(model, fov_up, fov_down, label_lut=lut, knn=None if arg.no_knn else KNN(), instances=clustering,
                       tta=tta, calibration=cal, mc_dropout=mcd)
  except ValueError as e:
    raise SystemExit(str(e))
  smap = None
  if arg.map:
    poses = kitti_lidar_poses(arg.poses, arg.calib)
    try:
      pose_of = np.array([scan_pose_index(f, len(poses)) for f in scans], np.int64)
      smap = SemanticMap(config.NUM_CLASS, voxel_size=arg.voxel_size, min_range=arg.map_min_range,
                         max_range=arg.map_max_range, ignore_class=config.CLASSES.index("None"))
    except ValueError as e:
      raise SystemExit(str(e))
    keep = Clustering().thing_ids(config) if arg.map_keep == "things" else ()
    scan_labels = []      # pass 1's point labels per batch, uint8 on the host

  def write_labels(files, labs):
    for f, lab in zip(files, labs):
      words = inv[lab] if inv is not None else lab.astype(np.uint32)
      words.astype(np.uint32).tofile(os.path.join(arg.output_dir, os.path.splitext(os.path.basename(f))[0] + ".label"))

  os.makedirs(arg.output_dir, exist_ok=True)
  loader = ScanBatchLoader(arg.format)
  for i in range(0, len(scans), arg.batch):
    files = scans[i:i + arg.batch]
    data = loader.load(files, labels[i:i + arg.batch] if labels is not None else None)
    if labels is not None:
      res = ev.update(data)
    else:
      res = ev.seg.segment_device(data["points"], data["offsets"], want_point_labels=True, knn=ev.knn,
                                  instances=clustering, tta=tta, confidence=cal.temperature if cal else None,
                                  mc_dropout=mcd)
    if cal is not None:
      pc = res["point_confidence"].cpu().numpy()
      for f, c in zip(files, np.split(pc, np.cumsum(data["sizes"])[:-1])):
        c.astype(np.float32).tofile(os.path.join(arg.output_dir, os.path.splitext(os.path.basename(f))[0] + ".conf"))
    if mcd is not None:
      mi = res["point_mi"].cpu().numpy()
      for f, u in zip(files, np.split(mi, np.cumsum(data["sizes"])[:-1])):
        u.astype(np.float32).tofile(os.path.join(arg.output_dir, os.path.splitext(os.path.basename(f))[0] + ".unc"))
    if clustering is not None:
      for f, words in zip(files, ev.seg.label_words(res, data["sizes"], inv)):
        words.tofile(os.path.join(arg.output_dir, os.path.splitext(os.path.basename(f))[0] + ".label"))
      continue
    if smap is not None:
      smap.vote(data["points"], data["offsets"], poses[pose_of[i:i + arg.batch]], res["point_labels"])
      scan_labels.append(res["point_labels"].cpu().numpy().astype(np.uint8))
      continue
    write_labels(files, ev.seg.point_labels(res, data["sizes"]))
  fused_iou = None
  if smap is not None:
    fused_iou = MeanIoU(num_classes=config.NUM_CLASS, name="MeanIoU") if labels is not None else None
    for j, i in enumerate(range(0, len(scans), arg.batch)):
      files = scans[i:i + arg.batch]
      data = loader.load(files, labels[i:i + arg.batch] if labels is not None else None)
      fused = smap.relabel(data["points"], data["offsets"], poses[pose_of[i:i + arg.batch]], scan_labels[j],
                           keep_classes=keep, min_votes=arg.map_min_votes)
      if fused_iou is not None:
        fused_iou.update_state(ev.ground_truth(data), fused)
      write_labels(files, np.split(fused.cpu().numpy(), np.cumsum(data["sizes"])[:-1]))
    print("semantic map: %d voxels of %g m" % (smap.num_voxels, smap.voxel_size))
    if arg.map_out:
      smap.save(arg.map_out)
  print("labelled %d scans -> %s" % (len(scans), arg.output_dir))
  if labels is None:
    return None
  rep = ev.finish()
  print_iou(rep, config.CLASSES)
  if rep["dropped"]:
    print("WARNING: %d of %d points have a ground-truth id that is not a class id (0 .. %d) and are not scored%s"
          % (rep["dropped"], int(rep["confusion_matrix"].sum()) + rep["dropped"], config.NUM_CLASS - 1,
             "" if arg.learning_map else "; pass --learning_map to map raw label ids to classes"))
  if clustering is not None and not kitti:
    print("no panoptic report: nuScenes lidarseg label files carry no instance ids")
  elif clustering is not None:
    print_panoptic(rep["panoptic"], config.CLASSES)
  if cal is not None:
    from .eval import print_reliability
    print_reliability(rep["calibration"]["reliability"], cal.temperature, "points")
  if mcd is not None:
    from .eval import print_mc_report
    print_mc_report(rep["mc_dropout"], "points")
  if fused_iou is not None:
    from .utils.util import confusion_matrix_to_iou_recall_precision
    cm = fused_iou.total_cm
    iou, recall, precision = confusion_matrix_to_iou_recall_precision(cm)
    rep["fused"] = dict(confusion_matrix=cm.cpu().numpy(), iou=iou, recall=recall, precision=precision,
                        miou=float(fused_iou.result()))
    print("FUSED (semantic map)")
    print_iou(rep["fused"], config.CLASSES)
  return rep


def print_iou(rep, class_names):
  """The per-class IoU / recall / precision lines and the mIoU of a report, in eval.py's format."""
  for c, cls in enumerate(class_names):
    print(cls.upper())
    print("IoU:       " + str(rep["iou"][c]))
    print("Recall:    " + str(rep["recall"][c]))
    print("Precision: " + str(rep["precision"][c]))
    print("")
  print("MIoU: {} ".format(rep["miou"]))


def print_panoptic(pan, class_names):
  """The PQ / SQ / RQ report of ``PanopticQuality.result()``, per thing class then the mean."""
  print("PANOPTIC (thing classes, point-wise)")
  for i, c in enumerate(pan["classes"]):
    print("%s PQ: %s SQ: %s RQ: %s (TP %d FP %d FN %d)%s" % (class_names[c].upper(), pan["pq"][i], pan["sq"][i],
                                                            pan["rq"][i], pan["tp"][i], pan["fp"][i], pan["fn"][i],
                                                            "" if pan["counted"][i] else " no segment"))
  print("PQ: {} SQ: {} RQ: {} ".format(pan["pq_mean"], pan["sq_mean"], pan["rq_mean"]))


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
  ap.add_argument("--instances", action="store_true", help="also an instance id per thing-class point (upper 16 bits)")
  ap.add_argument("--cluster_tau", type=float, default=0.5, help="metres: neighbouring points closer than this join")
  ap.add_argument("--cluster_rows", type=int, default=1, help="window half-height in rows (0..4)")
  ap.add_argument("--cluster_cols", type=int, default=2, help="window half-width in columns (0..8)")
  ap.add_argument("--min_points", type=int, default=10, help="instances with fewer points get id 0")
  ap.add_argument("--no_wrap", action="store_true", help="columns 0 and W-1 are not neighbours")
  ap.add_argument("--learning_map", default=None, help="yaml with `learning_map` / `learning_map_inv` (semantic-kitti.yaml)")
  from .tta import add_tta_flags
  add_tta_flags(ap)
  from .mc_dropout import add_mc_flags
  add_mc_flags(ap)
  from .calibration import add_temperature_flag
  ap.add_argument("--confidence", action="store_true", help="also write <name>.conf: float32 confidence per point")
  add_temperature_flag(ap)
  ap.add_argument("--bins", type=int, default=15, help="reliability bins of the --labels report (1..64)")
  ap.add_argument("--map", action="store_true", help="fuse the sequence's labels through a semantic voxel map (2 passes)")
  ap.add_argument("--poses", default=None, help="--map: the sequence's poses.txt (camera frame, 3x4 per line)")
  ap.add_argument("--calib", default=None, help="--map: the sequence's calib.txt (its Tr: line)")
  ap.add_argument("--voxel_size", type=float, default=0.2, help="--map: voxel edge in metres")
  ap.add_argument("--map_min_range", type=float, default=0.0, help="--map: nearer points cast no vote (metres)")
  ap.add_argument("--map_max_range", type=float, default=50.0, help="--map: farther points cast no vote; <= 0: no limit")
  ap.add_argument("--map_min_votes", type=int, default=1, help="--map: a voxel with fewer votes relabels nothing")
  ap.add_argument("--map_keep", choices=["things", "none"], default="things",
                  help="--map: points labelled as these classes keep their label")
  ap.add_argument("--map_out", default=None, help="--map: also write the map (.npz: voxels, counts, labels)")
  return segment_scans(ap.parse_args(argv))


if __name__ == "__main__":
  main()
