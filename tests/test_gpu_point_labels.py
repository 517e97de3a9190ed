"""Per-point labels on the GPU (pcls_point_labels, pcls_map_labels, ScanSegmenter / ScanEvaluator / segment_scans):
exact against the numpy oracle (oracle/point_labels.py) fed with the device's own scatter outputs, so every comparison
isolates the new kernels."""
import ctypes
import itertools
import os

import numpy as np
import pytest
import torch

from oracle import point_labels as PL
from tests.util import synth_scan

pytestmark = pytest.mark.gpu

H, W = 64, 512
GUARD = 0x5A5A5A5A      # guard band around the output: must stay untouched
SENTINEL = -12345       # prefill of the output: must not survive


def _lib():
  from pclsegmentation_b200 import _lib
  return _lib


def blocky_preds(rng, B, H, W, nc, noise=0.3):
  """Seeded, spatially blocky label map (4 x 8 blocks) with `noise` of the pixels relabelled at random: votes are
  contested."""
  blocks = rng.integers(0, nc, (B, (H + 3) // 4, (W + 7) // 8))
  p = np.repeat(np.repeat(blocks, 4, 1), 8, 2)[:, :H, :W]
  flip = rng.random(p.shape) < noise
  p[flip] = rng.integers(0, nc, int(flip.sum()))
  return p.astype(np.int32)


def edge_scan(rng, n=3000):
  """Points on rows 0 / H-1 and columns 0 / W-1 (pitch at the fov limits, yaw at +-pi), plus zero-xyz points."""
  r = rng.uniform(3, 60, n)
  k = np.arange(n) % 6
  pitch = np.where(k % 2 == 0, np.deg2rad(3.0 - 0.05), np.deg2rad(-25.0 + 0.05))
  pitch = np.where(k >= 4, np.deg2rad(rng.uniform(-24.0, 2.0, n)), pitch)
  yaw = np.where(k < 2, np.pi - 1e-4, np.where(k < 4, -np.pi + 1e-4, rng.choice([np.pi - 1e-4, -np.pi + 1e-4], n)))
  pts = np.stack([r * np.cos(pitch) * np.cos(yaw), r * np.cos(pitch) * np.sin(yaw), r * np.sin(pitch), rng.random(n)], 1)
  pts[::97, :3] = 0.0                                  # zero depth: dropped by the projection
  return pts.astype(np.float32)


def scatter(points, offsets, ring=None, H=H, W=W, fov_up=3.0, fov_down=-25.0):
  from pclsegmentation_b200.laserscan import SphericalProjector
  proj = SphericalProjector(H, W, fov_up, fov_down)
  return proj.project(points, offsets, ring=ring, want_image=False, want_idx=False, want_point_outputs=True)


def device_point_labels(preds, keys, offsets, px, py, ur, nc, none, search, k, weights, cutoff, ignore):
  """pcls_point_labels with the output inside a guard band (prefilled with a sentinel) and the scratch inside a guard
  band of empty words; checks both bands and returns the labels."""
  lib = _lib()
  B, Hh, Ww = preds.shape
  total = int(px.numel())
  g = 64
  buf = torch.full((total + 2 * g,), SENTINEL, dtype=torch.int32, device="cuda")
  buf[:g] = GUARD
  buf[g + total:] = GUARD
  out = buf[g:g + total]
  sbuf = torch.full((B * Hh * Ww + 2 * g,), -1, dtype=torch.int64, device="cuda")
  scratch = sbuf[g:g + B * Hh * Ww] if search > 1 else None
  w = None
  if weights is not None:
    w = (ctypes.c_float * len(weights))(*[float(v) for v in weights])
  lib.check(lib.load().pcls_point_labels(preds.data_ptr(), keys.data_ptr(), offsets.data_ptr(), B, Hh, Ww, total,
                                         px.data_ptr(), py.data_ptr(), ur.data_ptr(), nc, none, search, k, w,
                                         float(cutoff), ignore, scratch.data_ptr() if scratch is not None else None,
                                         out.data_ptr() if total else None, torch.cuda.current_stream().cuda_stream),
            "pcls_point_labels")
  host = buf.cpu().numpy()
  assert (host[:g] == GUARD).all() and (host[g + total:] == GUARD).all(), "guard band written"
  assert not (host[g:g + total] == SENTINEL).any(), "a point label was not written"
  s = sbuf.cpu().numpy()
  assert (s[:g] == -1).all() and (s[g + B * Hh * Ww:] == -1).all(), "scratch guard band written"
  return host[g:g + total]


def oracle_labels(preds_np, proj, offsets_np, nc, none, **kw):
  rng, valid = PL.winner_range(proj["keys"].cpu().numpy(), offsets_np, proj["unproj_range"].cpu().numpy())
  return PL.point_labels_batch(preds_np, rng, valid, offsets_np, proj["proj_x"].cpu().numpy(),
                               proj["proj_y"].cpu().numpy(), proj["unproj_range"].cpu().numpy(), nc, none, **kw)


@pytest.fixture(scope="module")
def batch():
  rng = np.random.default_rng(20261020)
  scans = [synth_scan(rng, 40000), np.zeros((0, 4), np.float32), synth_scan(rng, 1), edge_scan(rng),
           synth_scan(rng, 25000)]
  sizes = [s.shape[0] for s in scans]
  offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  pts = torch.from_numpy(np.concatenate(scans)).cuda()
  offsets = torch.from_numpy(offsets_np).cuda()
  proj = scatter(pts, offsets)
  px = proj["proj_x"].cpu().numpy()
  py = proj["proj_y"].cpu().numpy()
  lo, hi = offsets_np[3], offsets_np[4]
  e = slice(lo, hi)
  # the edge scan reaches every edge of the image and has dropped points
  assert (py[e] == 0).any() and (py[e] == H - 1).any() and (px[e] == 0).any() and (px[e] == W - 1).any()
  assert (px[e] < 0).any()
  # dense enough that most occupied pixels have losers
  occupied = int((proj["keys"][0] != -1).sum().item())
  assert 40000 - occupied > 0.3 * occupied
  return dict(offsets_np=offsets_np, offsets=offsets, pts=pts, proj=proj, rng=rng)


NONE_FOR = {11: 10, 20: 0, 32: 5}


def _cases():
  """search x k x cutoff x ignore, weights and num_classes cycled over the combinations (valid, distinct ones)."""
  out = [(1, 1, 0.0, -1, None, 20), (1, 1, 0.0, -1, None, 11), (1, 1, 0.0, -1, None, 32)]
  wsets = [None, 1.0, 2.0]
  ncs = [11, 20, 32]
  i = 0
  for s in (3, 5, 7, 9):
    for k in sorted({1, 5, min(s * s, 32)}):
      for cutoff, ign in itertools.product((0.0, 1.0, 0.05), ("off", "none", "frequent")):
        out.append((s, k, cutoff, ign, wsets[i % 3], ncs[(i // 3) % 3]))
        i += 1
  return out


@pytest.mark.parametrize("search", [1, 3, 5, 7, 9])
def test_kernel_equals_oracle(batch, search):
  offsets_np, proj = batch["offsets_np"], batch["proj"]
  B = len(offsets_np) - 1
  rng = np.random.default_rng(77 + search)
  preds = {nc: blocky_preds(rng, B, H, W, nc) for nc in (11, 20, 32)}
  dev = {nc: torch.from_numpy(p).cuda() for nc, p in preds.items()}
  n = 0
  for s, k, cutoff, ign, sigma, nc in _cases():
    if s != search:
      continue
    none = NONE_FOR[nc]
    if ign == "off" or ign == -1:
      ignore = -1
    elif ign == "none":
      ignore = none
    else:
      ignore = int(np.bincount(preds[nc].ravel(), minlength=nc).argmax())
    w = None if sigma is None else PL.window_weights(s, sigma)
    got = device_point_labels(dev[nc], proj["keys"], batch["offsets"], proj["proj_x"], proj["proj_y"],
                              proj["unproj_range"], nc, none, s, k, w, cutoff, ignore)
    want = oracle_labels(preds[nc], proj, offsets_np, nc, none, search=s, k=k, weights=w, cutoff=cutoff,
                         ignore_class=ignore)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, (s, k, cutoff, ignore, sigma, nc, bad[:10], got[bad[:10]], want[bad[:10]])
    n += 1
  assert n >= 3


def test_kernel_equals_oracle_on_quantized_ranges():
  """Hand-made scatter outputs with ranges on a 0.25 m grid: distances equal the cutoff and tie with each other on many
  points, so the tie rule and the cutoff at equality are exercised on the device, not only in the oracle."""
  rng = np.random.default_rng(31)
  B, Hq, Wq, n = 2, 16, 32, 1500
  px = rng.integers(0, Wq, B * n).astype(np.int32)
  py = rng.integers(0, Hq, B * n).astype(np.int32)
  px[::53], py[::53] = -1, -1
  ur = (2.0 + 0.25 * rng.integers(0, 16, B * n)).astype(np.float32)
  offsets_np = np.array([0, n, 2 * n], np.int64)
  keys = np.full((B, Hq, Wq), np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64)
  for i in range(B * n):                       # the scatter's rule: nearest point, then lowest index
    if px[i] < 0:
      continue
    b = i // n
    key = (np.uint64(ur[i:i + 1].view(np.uint32)[0]) << np.uint64(32)) | np.uint64(i - b * n)
    keys[b, py[i], px[i]] = min(keys[b, py[i], px[i]], key)
  preds = blocky_preds(rng, B, Hq, Wq, 11)
  d = {name: torch.from_numpy(a).cuda() for name, a in (("px", px), ("py", py), ("ur", ur), ("off", offsets_np),
                                                         ("keys", keys.view(np.int64)), ("preds", preds))}
  win, valid = PL.winner_range(keys.view(np.int64), offsets_np, ur)
  for s, k, cutoff, ign in ((3, 5, 1.0, -1), (3, 9, 0.5, 10), (5, 5, 0.25, -1), (5, 9, 1.0, 3), (7, 32, 0.5, -1)):
    got = device_point_labels(d["preds"], d["keys"], d["off"], d["px"], d["py"], d["ur"], 11, 10, s, k, None, cutoff,
                              ign)
    want = PL.point_labels_batch(preds, win, valid, offsets_np, px, py, ur, 11, 10, search=s, k=k, cutoff=cutoff,
                                 ignore_class=ign)
    assert np.array_equal(got, want), (s, k, cutoff, ign, np.flatnonzero(got != want)[:10])


def test_kernel_equals_oracle_on_ring_keys():
  """Ring projection: the keys carry ~index, not the depth, in the high word; the winner's range comes from
  unproj_range through the local index."""
  rng = np.random.default_rng(5)
  Hr, Wr = 32, 256
  scans = [synth_scan(rng, 12000, fov_up=10.0, fov_down=-30.0, rings=32), synth_scan(rng, 7000, fov_up=10.0,
                                                                                       fov_down=-30.0, rings=32)]
  rings = [rng.integers(0, Hr, s.shape[0]).astype(np.int32) for s in scans]
  sizes = [s.shape[0] for s in scans]
  offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  pts = torch.from_numpy(np.concatenate(scans)).cuda()
  offsets = torch.from_numpy(offsets_np).cuda()
  ring = torch.from_numpy(np.concatenate(rings)).cuda()
  proj = scatter(pts, offsets, ring=ring, H=Hr, W=Wr, fov_up=10.0, fov_down=-30.0)
  preds = blocky_preds(rng, 2, Hr, Wr, 11)
  for s, k, cutoff in ((3, 5, 1.0), (5, 5, 0.0), (5, 25, 1.0)):
    w = PL.window_weights(s, 1.0)
    got = device_point_labels(torch.from_numpy(preds).cuda(), proj["keys"], offsets, proj["proj_x"], proj["proj_y"],
                              proj["unproj_range"], 11, 10, s, k, w, cutoff, 10)
    want = oracle_labels(preds, proj, offsets_np, 11, 10, search=s, k=k, weights=w, cutoff=cutoff, ignore_class=10)
    assert np.array_equal(got, want), (s, k, cutoff, np.flatnonzero(got != want)[:10])


def _bench_scans():
  rng = np.random.default_rng(4321)         # the bench's projection leg
  sizes = rng.integers(115000, 125001, 64)
  return sizes, np.concatenate([synth_scan(rng, int(n)) for n in sizes])


def test_benchmark_size_against_oracle():
  """64 scans of 115-125 k points at 64 x 2048, predictions of a random-init SqueezeSegV2-KITTI forward: the defaults
  KNN() and search = 1 on every point of scans 0, 31 and 63."""
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map["squeezesegv2kitti"]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = 64, 2048
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(1)
  sizes, host = _bench_scans()
  pts = torch.from_numpy(host).cuda()
  offsets_np = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  offsets = torch.from_numpy(offsets_np).cuda()
  seg = ScanSegmenter(model, 3.0, -25.0)
  knn = KNN()
  res = seg.segment_device(pts, offsets, want_point_labels=True, knn=knn)
  plain = seg.segment_device(pts, offsets, want_point_labels=True)
  assert torch.equal(res["predictions"], plain["predictions"])
  preds = res["predictions"].cpu().numpy()
  assert len(np.unique(preds)) > 3, "the forward should produce several classes"
  proj = scatter(pts, offsets, H=64, W=2048)
  keys = proj["keys"].cpu().numpy()
  ur = proj["unproj_range"].cpu().numpy()
  px, py = proj["proj_x"].cpu().numpy(), proj["proj_y"].cpu().numpy()
  win, valid = PL.winner_range(keys, offsets_np, ur)
  got_knn, got_plain = res["point_labels"].cpu().numpy(), plain["point_labels"].cpu().numpy()
  none = mc.CLASSES.index("None")
  differ = 0
  for b in (0, 31, 63):
    sl = slice(offsets_np[b], offsets_np[b + 1])
    want = PL.point_labels(preds[b], win[b], valid[b], px[sl], py[sl], ur[sl], mc.NUM_CLASS, none, search=5, k=5,
                           weights=knn.weights(), cutoff=1.0, ignore_class=knn.ignore_index(mc))
    assert np.array_equal(got_knn[sl], want), (b, np.flatnonzero(got_knn[sl] != want)[:10])
    want1 = PL.point_labels(preds[b], win[b], valid[b], px[sl], py[sl], ur[sl], mc.NUM_CLASS, none)
    assert np.array_equal(got_plain[sl], want1), b
    differ += int((want != want1).sum())
  assert differ > 0, "the vote should change some labels at this density"
  model._release()


# ---- pipeline ----

@pytest.fixture(scope="module")
def small_model():
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map["squeezesegv2kitti"]()
  mc.AZIMUTH_LEVEL = 512
  model = model_map["squeezesegv2"](mc)
  model.randomize_batch_norm(2)
  return mc, model


def test_pipeline_paths_agree(small_model):
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  mc, model = small_model
  rng = np.random.default_rng(8)
  sizes = [20000, 0, 15000, 1]
  scans = [synth_scan(rng, n) for n in sizes]
  pts = torch.from_numpy(np.concatenate(scans)).cuda()
  offsets = torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).cuda()
  seg = ScanSegmenter(model, 3.0, -25.0)
  base = seg.segment_device(pts, offsets, want_logits=True)
  assert "point_labels" not in base
  for knn in (None, KNN(), KNN(search=3, k=9, sigma=2.0, cutoff=0.0, ignore_class=-1)):
    one = seg.segment_device(pts, offsets, want_logits=True, want_point_labels=True, knn=knn)
    two = seg.segment_device(pts, offsets, want_logits=True, want_image=True, want_point_labels=True, knn=knn)
    assert one["point_labels"].dtype == torch.int32 and one["point_labels"].shape == (sum(sizes),)
    assert torch.equal(one["point_labels"], two["point_labels"])
    assert torch.equal(one["predictions"], base["predictions"]) and torch.equal(one["logits"], base["logits"])
    assert torch.equal(two["predictions"], base["predictions"]) and torch.equal(two["logits"], base["logits"])
  # search = 1 is the gather predictions[b, py, px] for every projected point
  plain = seg.segment_device(pts, offsets, want_point_labels=True)
  proj = scatter(pts, offsets)
  px, py = proj["proj_x"].long(), proj["proj_y"].long()
  b = torch.repeat_interleave(torch.arange(len(sizes), device="cuda"), torch.as_tensor(sizes, device="cuda"))
  ok = px >= 0
  assert ok.sum() > 0.99 * sum(sizes)
  gathered = plain["predictions"][b[ok], py[ok], px[ok]]
  assert torch.equal(plain["point_labels"][ok], gathered)
  assert (plain["point_labels"][~ok] == mc.CLASSES.index("None")).all()
  parts = seg.point_labels(plain, sizes)
  assert [p.shape[0] for p in parts] == sizes and all(p.dtype == np.int32 for p in parts)
  assert np.array_equal(np.concatenate(parts), plain["point_labels"].cpu().numpy())
  res = seg.segment(scans, want_point_labels=True, knn=KNN())
  assert torch.equal(res["point_labels"], seg.segment_device(pts, offsets, want_point_labels=True,
                                                              knn=KNN())["point_labels"])


# ---- point-wise evaluation ----

def test_map_labels_equals_numpy():
  lib = _lib()
  rng = np.random.default_rng(3)
  words = rng.integers(0, 2 ** 32, 10007, dtype=np.uint64).astype(np.uint32)
  words[:3000] = (words[:3000] & 0xFFFF0000) | rng.integers(0, 40, 3000).astype(np.uint32)
  lut = rng.integers(0, 20, 35).astype(np.int32)
  d_words = torch.from_numpy(words.view(np.int32)).cuda()
  out = torch.empty(words.shape[0], dtype=torch.int32, device="cuda")
  s = torch.cuda.current_stream().cuda_stream
  sem = (words & 0xFFFF).astype(np.int64)
  lib.check(lib.load().pcls_map_labels(d_words.data_ptr(), words.shape[0], torch.from_numpy(lut).cuda().data_ptr(),
                                       lut.shape[0], out.data_ptr(), s), "pcls_map_labels")
  want = np.where(sem < lut.shape[0], lut[np.minimum(sem, lut.shape[0] - 1)], 0)
  assert np.array_equal(out.cpu().numpy(), want)
  assert (sem >= lut.shape[0]).any() and (sem < lut.shape[0]).any()
  lib.check(lib.load().pcls_map_labels(d_words.data_ptr(), words.shape[0], None, 0, out.data_ptr(), s), "pcls_map_labels")
  assert np.array_equal(out.cpu().numpy(), sem)


def _write_dataset(tmp_path, fmt, rng, sizes, H=64, fov_up=3.0, fov_down=-25.0):
  scan_dir, lab_dir = tmp_path / "velodyne", tmp_path / "labels"
  scan_dir.mkdir()
  lab_dir.mkdir()
  scans, words = [], []
  for i, n in enumerate(sizes):
    s = synth_scan(rng, n, fov_up=fov_up, fov_down=fov_down, rings=H)
    if fmt == "kitti":
      s.tofile(str(scan_dir / ("%06d.bin" % i)))
      w = (rng.integers(0, 300, n).astype(np.uint32) << 16) | rng.choice([0, 10, 11, 40, 44, 48, 50, 70, 252, 999], n).astype(np.uint32)
      w.astype(np.uint32).tofile(str(lab_dir / ("%06d.label" % i)))
    else:
      rec = np.concatenate([s, rng.integers(0, H, (n, 1)).astype(np.float32)], 1)
      rec.astype(np.float32).tofile(str(scan_dir / ("%06d.bin" % i)))
      w = rng.integers(0, 32, n).astype(np.uint8)
      w.tofile(str(lab_dir / ("%06d.bin" % i)))
      w = w.astype(np.uint32)
    scans.append(s)
    words.append(w)
  return scan_dir, lab_dir, scans, words


@pytest.mark.parametrize("fmt", ["kitti", "nuscenes"])
def test_scan_evaluator_matrix(tmp_path, small_model, fmt):
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  mc, model = small_model
  rng = np.random.default_rng(11)
  fu, fd = (3.0, -25.0) if fmt == "kitti" else (12.0, -30.0)
  sizes = [9000, 7000, 5000]
  scan_dir, lab_dir, scans, words = _write_dataset(tmp_path, fmt, rng, sizes, fov_up=fu, fov_down=fd)
  lut = np.zeros(260, np.int32)
  lut[[10, 11, 40, 44, 48, 50, 70, 252]] = [1, 2, 9, 10, 11, 13, 15, 1]
  lut[:32] = np.where(np.arange(32) % 3 == 0, np.arange(32) % mc.NUM_CLASS, lut[:32])
  ext = ".label" if fmt == "kitti" else ".bin"
  files = sorted(str(p) for p in scan_dir.iterdir())
  labs = sorted(str(p) for p in lab_dir.iterdir() if p.name.endswith(ext))
  loader = ScanBatchLoader(fmt)
  knn = KNN()
  ev = ScanEvaluator(model, fu, fd, label_lut=lut, knn=knn)
  cm = np.zeros((mc.NUM_CLASS, mc.NUM_CLASS), np.int64)
  for lo in (0, 2):
    fs = files[lo:lo + 2]
    data = loader.load(fs, labs[lo:lo + 2])
    res = ev.update(data)
    proj = scatter(data["points"], data["offsets"], fov_up=fu, fov_down=fd)
    offs = data["offsets"].cpu().numpy()
    want = oracle_labels(res["predictions"].cpu().numpy(), proj, offs, mc.NUM_CLASS, mc.CLASSES.index("None"),
                         search=5, k=5, weights=knn.weights(), cutoff=1.0, ignore_class=knn.ignore_index(mc))
    w = np.concatenate(words[lo:lo + 2]).astype(np.int64) & 0xFFFF
    gt = np.where(w < lut.shape[0], lut[np.minimum(w, lut.shape[0] - 1)], 0)
    assert np.array_equal(res["gt"].cpu().numpy(), gt)
    cm += np.bincount(gt * mc.NUM_CLASS + want, minlength=mc.NUM_CLASS ** 2).reshape(mc.NUM_CLASS, mc.NUM_CLASS)
  rep = ev.finish()
  assert np.array_equal(rep["confusion_matrix"], cm) and cm.sum() == sum(sizes)
  from oracle import confusion as C
  assert abs(rep["miou"] - C.mean_iou(cm)) < 1e-6


# ---- CLI ----

def test_segment_scans_cli(tmp_path, capsys):
  import yaml
  from pclsegmentation_b200 import segment_scans
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader, learning_map_lut
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  from pclsegmentation_b200.utils.args_loader import load_model_config
  rng = np.random.default_rng(12)
  sizes = [8000, 6000, 7000]
  scan_dir, lab_dir, scans, words = _write_dataset(tmp_path, "kitti", rng, sizes)
  raw = [0, 10, 11, 40, 44, 48, 50, 70, 252, 999]
  learning_map = {r: i % 20 for i, r in enumerate(raw)}
  learning_map_inv = {c: 1000 + 7 * c for c in range(20)}
  ypath = tmp_path / "map.yaml"
  ypath.write_text(yaml.safe_dump({"learning_map": learning_map, "learning_map_inv": learning_map_inv}))
  out = tmp_path / "pred"
  args = ["--scans", str(scan_dir / "*.bin"), "--format", "kitti", "-m", "squeezesegv2", "-n", "squeezesegv2kitti",
          "--random_init", "--batch", "2", "--output_dir", str(out), "--learning_map", str(ypath)]
  segment_scans.main(args)
  mc, model = load_model_config("squeezesegv2", "squeezesegv2kitti")     # the CLI's model: same seeded init
  ev = ScanEvaluator(model, 3.0, -25.0, label_lut=learning_map_lut(learning_map), knn=KNN())
  loader = ScanBatchLoader("kitti")
  files = sorted(str(p) for p in scan_dir.iterdir())
  labs = sorted(str(p) for p in lab_dir.iterdir())
  inv = learning_map_lut(learning_map_inv)
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2], labs[lo:lo + 2])
    res = ev.update(data)
    for f, lab in zip(files[lo:lo + 2], ev.seg.point_labels(res, data["sizes"])):
      got = np.fromfile(str(out / (os.path.splitext(os.path.basename(f))[0] + ".label")), dtype=np.uint32)
      assert got.shape == lab.shape
      assert np.array_equal(got, inv[lab].astype(np.uint32))
  rep = ev.finish()
  capsys.readouterr()
  rep_cli = segment_scans.main(args + ["--labels", str(lab_dir / "*.label")])
  printed = capsys.readouterr().out
  assert "MIoU: {} ".format(rep["miou"]) in printed and "CAR" in printed
  assert np.array_equal(rep_cli["confusion_matrix"], rep["confusion_matrix"])
  assert rep_cli["dropped"] == 0 and "WARNING" not in printed
  # raw ids without --learning_map: ids >= NUM_CLASS (10, 40, ..., 999) are counted as unscored and reported
  raw_args = [a for a in args if a not in ("--learning_map", str(ypath))]
  rep_raw = segment_scans.main(raw_args + ["--labels", str(lab_dir / "*.label"), "--output_dir", str(tmp_path / "raw")])
  printed = capsys.readouterr().out
  w = np.concatenate(words).astype(np.int64) & 0xFFFF
  assert rep_raw["dropped"] == int((w >= mc.NUM_CLASS).sum()) > 0
  assert int(rep_raw["confusion_matrix"].sum()) == int((w < mc.NUM_CLASS).sum())
  assert "WARNING: %d of %d points" % (rep_raw["dropped"], sum(sizes)) in printed and "--learning_map" in printed
  # --no_knn: each point takes its pixel's label
  segment_scans.main(args + ["--no_knn", "--output_dir", str(tmp_path / "plain")])
  ev1 = ScanEvaluator(model, 3.0, -25.0)
  data = loader.load(files[:2])
  res = ev1.seg.segment_device(data["points"], data["offsets"], want_point_labels=True)
  lab = ev1.seg.point_labels(res, data["sizes"])[0]
  got = np.fromfile(str(tmp_path / "plain" / (os.path.splitext(os.path.basename(files[0]))[0] + ".label")), np.uint32)
  assert np.array_equal(got, inv[lab].astype(np.uint32))
