"""Calibrated confidence on the GPU (pcls_confidence, pcls_temperature_nll, pcls_reliability_update,
pcls_point_confidence and their pipelines / CLIs) against the float64 oracle (oracle/calibration.py), the head's own bits
and the paths without calibration."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import calibration as O
from tests.util import synth_range_images, synth_scan

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
  from pclsegmentation_b200 import _lib
  return _lib


def _s():
  return torch.cuda.current_stream().cuda_stream


def _f32(v):
  return (ctypes.c_float * len(v))(*[float(x) for x in v])


def device_confidence(src, nc, a, mask=None, probs_mode=False):
  """pcls_confidence with every output -> (probs, conf, entropy) numpy."""
  lib = _lib()
  n = src.numel() // nc
  p = torch.full((n, nc), -7.0, dtype=torch.float32, device="cuda")
  c = torch.full((n,), -7.0, dtype=torch.float32, device="cuda")
  e = torch.full((n,), -7.0, dtype=torch.float32, device="cuda")
  lib.check(lib.load().pcls_confidence(None if probs_mode else src.data_ptr(), src.data_ptr() if probs_mode else None,
                                       mask.data_ptr() if mask is not None else None, n, nc, float(a), p.data_ptr(),
                                       c.data_ptr(), e.data_ptr(), _s()), "pcls_confidence")
  return p.cpu().numpy(), c.cpu().numpy(), e.cpu().numpy()


def softmax_bound(z, a):
  """Per row, a bound on |p_fl32 - p| / p of the float32 softmax of z * a: s and m carry u S, s - m 4 u S, expf 2 ulp,
  the NC-term sum NC u, the division 1 ulp: u (8 S + 2 NC + 8) with S = max |s| (doubled: the sum's error enters p
  through the denominator as well)."""
  S = np.abs(z.astype(np.float64) * np.float64(a)).max(1)
  nc = z.shape[1]
  return U * (8 * S + 2 * nc + 8) * 2


@pytest.mark.parametrize("nc", [11, 20, 32])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 2 ** 20 + 7])
def test_confidence_at_t1_is_the_head_bit_for_bit(nc, n):
  lib = _lib()
  rng = np.random.default_rng(nc * 7 + n % 97)
  z = rng.normal(0, 4, (n, nc)).astype(np.float32)
  z[0, :] = 1.5                                            # all classes tie
  mask = (rng.random(n) < 0.8).astype(np.uint8)
  dz, dm = torch.from_numpy(z).cuda(), torch.from_numpy(mask).cuda()
  hp = torch.empty((n, nc), dtype=torch.float32, device="cuda")
  hy = torch.empty(n, dtype=torch.int32, device="cuda")
  lib.check(lib.load().pcls_head(dz.data_ptr(), dm.data_ptr(), n, nc, nc - 1, hp.data_ptr(), hy.data_ptr(), _s()),
            "pcls_head")
  p, c, e = device_confidence(dz, nc, 1.0, dm)
  hp = hp.cpu().numpy()
  assert np.array_equal(p.view(np.uint32), hp.view(np.uint32))
  want_c = np.where(mask != 0, hp.max(1), np.float32(0))
  assert np.array_equal(c.view(np.uint32), want_c.view(np.uint32))
  _, oc, oe = O.confidence(logits=z, mask=mask)
  eps = softmax_bound(z, 1.0)
  tol = (eps * (np.log(nc) + 1) + 4 * nc * U) / np.log(nc)
  assert (np.abs(e - oe) <= tol).all(), np.abs(e - oe).max()
  assert np.all(e[mask == 0] == 0) and (e[mask != 0] > 0).all()
  # probs mode over the head's probabilities: the same confidence, the probabilities copied
  p2, c2, e2 = device_confidence(torch.from_numpy(hp).cuda(), nc, 1.0, dm, probs_mode=True)
  assert np.array_equal(p2.view(np.uint32), hp.view(np.uint32)) and np.array_equal(c2.view(np.uint32), c.view(np.uint32))
  assert np.array_equal(e2.view(np.uint32), e.view(np.uint32))


@pytest.mark.parametrize("T", [0.5, 2.0, 3.7])
@pytest.mark.parametrize("nc", [11, 20, 32])
def test_tempered_confidence_against_float64(T, nc):
  rng = np.random.default_rng(int(T * 10) + nc)
  n = 100_003
  z = rng.normal(0, 4, (n, nc)).astype(np.float32)
  a = O.inv_temperature(T)
  p, c, e = device_confidence(torch.from_numpy(z).cuda(), nc, a)
  op, oc, oe = O.confidence(logits=z, a=a)
  eps = softmax_bound(z, a)
  assert (np.abs(p - op) <= eps[:, None] * op + 1e-45).all(), (np.abs(p - op) / op).max()
  assert (np.abs(c - oc) <= eps * oc).all()
  tol = (eps * (np.log(nc) + 1) + 4 * nc * U) / np.log(nc)
  assert (np.abs(e - oe) <= tol).all(), np.abs(e - oe).max()
  # the argmax does not depend on T: conf sits at the head's class
  _, c1, _ = device_confidence(torch.from_numpy(z).cuda(), nc, 1.0)
  assert (c <= c1 * (1 + eps)).all() if T > 1 else (c >= c1 * (1 - eps)).all()


@pytest.mark.parametrize("n_temps", [1, 17, 64])
def test_temperature_nll_against_float64(n_temps):
  lib = _lib()
  rng = np.random.default_rng(n_temps)
  n, nc, ignore = 300_017, 20, 19
  z = rng.normal(0, 4, (n, nc)).astype(np.float32)
  label = rng.integers(-3, nc + 3, n).astype(np.int32)
  label[::11] = ignore
  temps = np.exp(rng.uniform(np.log(0.25), np.log(4.0), n_temps))
  inv = [O.inv_temperature(T) for T in temps]
  acc = torch.zeros(n_temps, dtype=torch.float64, device="cuda")
  cnt = torch.zeros(1, dtype=torch.int64, device="cuda")
  dz, dl = torch.from_numpy(z).cuda(), torch.from_numpy(label).cuda()
  for _ in range(2):                                       # accumulated in place
    lib.check(lib.load().pcls_temperature_nll(dz.data_ptr(), dl.data_ptr(), n, nc, ignore, n_temps, _f32(inv),
                                              acc.data_ptr(), cnt.data_ptr(), _s()), "pcls_temperature_nll")
  sums, count, bound = O.temperature_nll(z, label, nc, ignore, inv)
  assert int(cnt.item()) == 2 * count and count == ((label >= 0) & (label < nc) & (label != ignore)).sum()
  got = acc.cpu().numpy() / 2
  assert (np.abs(got - sums) <= bound).all(), (np.abs(got - sums) / bound).max()


def test_planted_temperature_fit_on_the_gpu():
  from pclsegmentation_b200.calibration import Calibration, TemperatureNLL
  rng = np.random.default_rng(5)
  n, nc = 2 ** 20, 20
  for T0 in (0.5, 2.0):
    z = rng.normal(0, 3, (n, nc)).astype(np.float32)
    p = O.softmax(z, O.inv_temperature(T0))
    label = (rng.random(n)[:, None] > np.cumsum(p, 1)).sum(1).clip(0, nc - 1).astype(np.int32)
    nll = TemperatureNLL(Calibration(fit=True), nc, -1)
    nll.update(torch.from_numpy(z).cuda(), torch.from_numpy(label).cuda())
    r = nll.result()
    assert r["counted"] == n and not r["at_edge"] and abs(r["t_star"] / T0 - 1) < 0.02, r["t_star"]
    assert len(r["temperatures"]) == 64 and r["nll_at_1"] >= r["nll"].min() - 1e-9


@pytest.mark.parametrize("n_bins", [1, 15, 64])
def test_reliability_counts_exact(n_bins):
  lib = _lib()
  rng = np.random.default_rng(n_bins)
  n, nc = 1_000_003, 20
  conf = rng.random(n).astype(np.float32)
  conf[::5] = (rng.integers(0, n_bins + 1, conf[::5].size) / n_bins).astype(np.float32)   # exactly on bin edges
  pred = rng.integers(-1, nc + 1, n).astype(np.int32)
  label = np.where(rng.random(n) < 0.5, pred, rng.integers(-2, nc + 2, n)).astype(np.int32)
  cnt = torch.zeros(n_bins, dtype=torch.int64, device="cuda")
  cor = torch.zeros(n_bins, dtype=torch.int64, device="cuda")
  cs = torch.zeros(n_bins, dtype=torch.float64, device="cuda")
  d = [torch.from_numpy(v).cuda() for v in (conf, pred, label)]
  lib.check(lib.load().pcls_reliability_update(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), n, nc, 3, n_bins,
                                               cnt.data_ptr(), cor.data_ptr(), cs.data_ptr(), _s()),
            "pcls_reliability_update")
  wc, wr, ws = O.reliability(conf, pred, label, nc, 3, n_bins)
  assert np.array_equal(cnt.cpu().numpy(), wc) and np.array_equal(cor.cpu().numpy(), wr)
  assert np.allclose(cs.cpu().numpy(), ws, rtol=1e-12, atol=0)
  assert wc.sum() > n // 3


def test_point_confidence_exact_gather():
  lib = _lib()
  rng = np.random.default_rng(6)
  B, H, W, nc = 3, 8, 64, 20
  probs = rng.random((B, H, W, nc)).astype(np.float32)
  sizes = [5000, 0, 7001]
  offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
  total = int(offsets[-1])
  px = rng.integers(0, W, total).astype(np.int32)
  py = rng.integers(0, H, total).astype(np.int32)
  px[::13] = -1
  py[::13] = -1
  lab = rng.integers(-2, nc + 2, total).astype(np.int32)
  out = torch.full((total + 64,), 1e30, dtype=torch.float32, device="cuda")
  d = [torch.from_numpy(v).cuda() for v in (probs, offsets, px, py, lab)]
  lib.check(lib.load().pcls_point_confidence(d[0].data_ptr(), d[1].data_ptr(), B, H, W, total, d[2].data_ptr(),
                                             d[3].data_ptr(), d[4].data_ptr(), nc, out.data_ptr(), _s()),
            "pcls_point_confidence")
  got = out.cpu().numpy()
  want = O.point_confidence(probs, offsets, px, py, lab)
  assert np.array_equal(got[:total].view(np.uint32), want.view(np.uint32)) and (got[total:] == np.float32(1e30)).all()
  assert (want[px < 0] == 0).all() and (want[(lab < 0) | (lab >= nc)] == 0).all()


# ---- pipelines ----

def _model(name="squeezesegv2", cfg="squeezesegv2kitti", W=256, prec=0, seed=1):
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map[cfg]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = 64, W
  model = model_map[name](mc)
  model.precision = prec
  model.randomize_batch_norm(seed)
  return mc, model


@pytest.mark.parametrize("name,cfg,prec", [("squeezesegv2", "squeezesegv2kitti", 0), ("squeezesegv2", "squeezesegv2kitti", 1),
                                           ("darknet21", "darknet21", 0)])
def test_evaluator_with_calibration(name, cfg, prec):
  from pclsegmentation_b200.calibration import Calibration, confidence
  from pclsegmentation_b200.metrics import reliability_scores
  from pclsegmentation_b200.pipeline import Evaluator
  mc, model = _model(name, cfg, prec=prec)
  nc, none = mc.NUM_CLASS, mc.CLASSES.index("None")
  frames = synth_range_images(np.random.default_rng(3), 6, 64, 256, channels=6, num_classes=nc)
  cal = Calibration(temperature=1.7, n_bins=15, fit=True, grid=(0.3, 3.0, 17))
  plain, ev = Evaluator(model), Evaluator(model, calibration=cal)
  cnt, cor, cs = np.zeros(15, np.int64), np.zeros(15, np.int64), np.zeros(15)
  temps = np.concatenate([cal.grid_temperatures(), [1.0, 1.7]])
  sums, count, bound = np.zeros(temps.size), 0, np.zeros(temps.size)
  for lo in (0, 4):
    x = frames[lo:lo + 4]
    want_y = plain.update(x)
    y, label = ev.update(x, return_label=True)
    assert torch.equal(y, want_y)
    logits = model.forward_device(torch.from_numpy(x).cuda(), None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD,
                                  want_logits=True)["logits"]
    conf = confidence(nc, logits=logits, temperature=1.7)["confidence"].cpu().numpy()
    a, b, c = O.reliability(conf, y.cpu().numpy(), label.cpu().numpy(), nc, none, 15)
    cnt, cor, cs = cnt + a, cor + b, cs + c
    s, k, bd = O.temperature_nll(logits.cpu().numpy(), label.cpu().numpy(), nc, none,
                                 [O.inv_temperature(T) for T in temps])
    sums, count, bound = sums + s, count + k, bound + bd
  rp, rc = plain.finish(), ev.finish()
  assert np.array_equal(rp["confusion_matrix"], rc["confusion_matrix"]) and "calibration" not in rp
  rel, nll = rc["calibration"]["reliability"], rc["calibration"]["nll"]
  want = reliability_scores(cnt, cor, cs)
  assert np.array_equal(rel["bin_count"], cnt) and np.array_equal(rel["bin_accuracy"], want["bin_accuracy"])
  assert np.allclose(rel["bin_confidence"], want["bin_confidence"], rtol=1e-12, atol=0)
  assert rel["ece"] == pytest.approx(want["ece"], rel=1e-12)
  assert rel["count"] == cnt.sum() > 0 and nll["counted"] == count
  got = np.concatenate([nll["nll"], [nll["nll_at_1"], nll["nll_at_temperature"]]]) * count
  assert (np.abs(got - sums) <= bound + 1e-9 * np.abs(sums)).all()
  model._release()


@pytest.fixture(scope="module")
def scan_model():
  return _model(W=512, seed=2)


def _scans(rng, sizes):
  pts = [synth_scan(rng, n) for n in sizes]
  return (torch.from_numpy(np.concatenate(pts)).cuda(),
          torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).cuda())


@pytest.mark.parametrize("T", [1.0, 2.0])
def test_segment_device_confidence(scan_model, T):
  from pclsegmentation_b200.calibration import confidence
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  mc, model = scan_model
  pts, offsets = _scans(np.random.default_rng(9), [20000, 0, 15000, 1])
  seg = ScanSegmenter(model, 3.0, -25.0)
  plain = seg.segment_device(pts, offsets, want_point_labels=True, knn=KNN())
  for want_image in (False, True):                         # staged and materialised routes
    res = seg.segment_device(pts, offsets, want_point_labels=True, knn=KNN(), confidence=T, want_image=want_image)
    assert torch.equal(res["predictions"], plain["predictions"]) and torch.equal(res["point_labels"], plain["point_labels"])
    assert "probabilities" not in res and "logits" not in res
    full = seg.segment_device(pts, offsets, want_point_labels=True, knn=KNN(), want_logits=True, want_probabilities=True)
    proj = seg.projector.project(pts, offsets, empty_fill=0.0, want_point_outputs=True)
    mask = (proj["proj_idx"] >= 0).to(torch.uint8)
    if T == 1.0:                                           # the forward's own probabilities (the fused head's bits)
      c = confidence(mc.NUM_CLASS, probs=full["probabilities"], mask=mask)
      probs = full["probabilities"]
    else:
      c = confidence(mc.NUM_CLASS, logits=full["logits"], mask=mask, temperature=T, want_probs=True)
      probs = c["probabilities"]
    assert torch.equal(res["confidence"], c["confidence"])
    want = O.point_confidence(probs.cpu().numpy(), offsets.cpu().numpy(), proj["proj_x"].cpu().numpy(),
                              proj["proj_y"].cpu().numpy(), res["point_labels"].cpu().numpy())
    assert np.array_equal(res["point_confidence"].cpu().numpy(), want)
    assert (res["confidence"][mask == 0] == 0).all() and (res["confidence"][mask != 0] > 0).all()
  with pytest.raises(ValueError, match="point labels"):
    seg.segment_device(pts, offsets, confidence=T)


@pytest.mark.parametrize("T", [1.0, 2.0])
def test_scan_evaluator_with_calibration(tmp_path, scan_model, T):
  from pclsegmentation_b200.calibration import Calibration
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  from pclsegmentation_b200.tta import TTA
  mc, model = scan_model
  rng = np.random.default_rng(11)
  files, labs = _write_kitti(tmp_path, rng, [9000, 7000, 5000])
  ev = ScanEvaluator(model, 3.0, -25.0, knn=KNN(), calibration=Calibration(temperature=T, n_bins=10))
  loader = ScanBatchLoader("kitti")
  cnt, cor, cs = np.zeros(10, np.int64), np.zeros(10, np.int64), np.zeros(10)
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2], labs[lo:lo + 2])
    res = ev.update(data)
    want = ev.seg.segment_device(data["points"], data["offsets"], want_point_labels=True, knn=KNN(), confidence=T)
    assert torch.equal(res["point_confidence"], want["point_confidence"])
    a, b, c = O.reliability(res["point_confidence"].cpu().numpy(), res["point_labels"].cpu().numpy(),
                            res["gt"].cpu().numpy(), mc.NUM_CLASS, mc.CLASSES.index("None"), 10)
    cnt, cor, cs = cnt + a, cor + b, cs + c
  rel = ev.finish()["calibration"]["reliability"]
  assert np.array_equal(rel["bin_count"], cnt) and rel["count"] > 0
  assert rel["ece"] == pytest.approx(O.ece_mce(cnt, cor, cs)[0], rel=1e-12)
  with pytest.raises(ValueError, match="merges probabilities"):
    ScanEvaluator(model, calibration=Calibration(temperature=2.0), tta=TTA())
  with pytest.raises(ValueError, match="fitted on pixels"):
    ScanEvaluator(model, calibration=Calibration(fit=True))


def test_tta_confidence_comes_from_the_merged_probabilities(scan_model):
  from pclsegmentation_b200.calibration import Calibration, confidence
  from pclsegmentation_b200.pipeline import Evaluator
  from pclsegmentation_b200.tta import TTA, forward_tta
  mc, model = scan_model
  frames = synth_range_images(np.random.default_rng(4), 2, 64, 512, channels=6, num_classes=mc.NUM_CLASS)
  tta = TTA(shifts=(0, 128))
  ev = Evaluator(model, tta=tta, calibration=Calibration())
  y, label = ev.update(frames, return_label=True)
  merged = forward_tta(model, torch.from_numpy(frames).cuda(), tta, want_probabilities=True)
  assert torch.equal(y, merged["predictions"])
  conf = confidence(mc.NUM_CLASS, probs=merged["probabilities"])["confidence"].cpu().numpy()
  cnt, _, _ = O.reliability(conf, y.cpu().numpy(), label.cpu().numpy(), mc.NUM_CLASS, mc.CLASSES.index("None"), 15)
  rep = ev.finish()["calibration"]
  assert np.array_equal(rep["reliability"]["bin_count"], cnt) and rep["nll"] is None
  for cal in (Calibration(temperature=2.0), Calibration(fit=True)):
    with pytest.raises(ValueError, match="merges probabilities"):
      Evaluator(model, tta=tta, calibration=cal)


# ---- CLIs ----

def _write_kitti(tmp_path, rng, sizes):
  scan_dir, lab_dir = tmp_path / "velodyne", tmp_path / "labels"
  scan_dir.mkdir()
  lab_dir.mkdir()
  for i, n in enumerate(sizes):
    synth_scan(rng, n).tofile(str(scan_dir / ("%06d.bin" % i)))
    rng.integers(0, 11, n).astype(np.uint32).tofile(str(lab_dir / ("%06d.label" % i)))
  return sorted(str(p) for p in scan_dir.iterdir()), sorted(str(p) for p in lab_dir.iterdir())


@pytest.fixture(scope="module")
def golden(golden_dir):
  with np.load(os.path.join(golden_dir, "nn_sample_dataset.npz")) as f:
    return {k: f[k] for k in f.files}


def test_inference_and_eval_cli_calibration(tmp_path, golden, capsys):
  from pclsegmentation_b200 import eval as ev
  from pclsegmentation_b200 import inference
  from pclsegmentation_b200.calibration import confidence, raw_mask
  from pclsegmentation_b200.utils.args_loader import load_model_config
  mc, model = load_model_config("squeezesegv2", "squeezesegv2")
  model.randomize_batch_norm(1)
  wpath = str(tmp_path / "weights.npz")
  model.save_weights_npz(wpath)
  d = tmp_path / "data" / "val"
  d.mkdir(parents=True)
  for n, f in zip(golden["names"], golden["frames"]):
    np.save(str(d / str(n)), f.astype(np.float64))
  frames = torch.from_numpy(golden["frames"].astype(np.float32)).cuda()
  res = model.forward_device(frames, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_logits=True)
  want = confidence(mc.NUM_CLASS, logits=res["logits"], mask=raw_mask(frames, mc), temperature=1.5)["confidence"]
  want = want.cpu().numpy()
  out = tmp_path / "out"
  inference.main(["-d", str(d / "*.npy"), "-m", "squeezesegv2", "-n", "squeezesegv2", "-t", str(out), "-p", wpath,
                  "-b", "2", "--no_plots", "--confidence", "--temperature", "1.5"])
  for i, n in enumerate(golden["names"]):
    stem = os.path.splitext(str(n))[0]
    got = np.load(str(out / ("conf_" + stem + ".npy")))
    assert got.dtype == np.float32 and np.array_equal(got, want[i])
    assert np.array_equal(np.load(str(out / ("pred_" + stem + ".npy"))), res["predictions"][i].cpu().numpy())
  capsys.readouterr()
  js = str(tmp_path / "cal.json")
  rep = ev.main(["-d", str(tmp_path / "data"), "-i", "val", "-m", "squeezesegv2", "-n", "squeezesegv2", "-p", wpath,
                 "-b", "2", "--calibration", "--fit_temperature", "--calibration_json", js])
  text = capsys.readouterr().out
  assert text.index("MIoU:") < text.index("RELIABILITY") < text.index("T*:") and "NLL(1):" in text and "ECE:" in text
  with open(js) as f:
    back = json.load(f)
  cal = rep["calibration"]
  assert back["reliability"]["bin_count"] == cal["reliability"]["bin_count"].tolist()
  assert back["nll"]["t_star"] == cal["nll"]["t_star"] and back["fitted"]["temperature"] == cal["nll"]["t_star"]
  assert back["reliability"]["ece"] == cal["reliability"]["ece"]
  plain = ev.main(["-d", str(tmp_path / "data"), "-i", "val", "-m", "squeezesegv2", "-n", "squeezesegv2", "-p", wpath,
                   "-b", "2"])
  assert np.array_equal(plain["confusion_matrix"], rep["confusion_matrix"]) and "calibration" not in plain


def test_segment_scans_cli_confidence(tmp_path, capsys):
  from pclsegmentation_b200 import segment_scans
  from pclsegmentation_b200.calibration import Calibration
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  from pclsegmentation_b200.utils.args_loader import load_model_config
  files, labs = _write_kitti(tmp_path, np.random.default_rng(12), [8000, 6000, 7000])
  out = tmp_path / "pred"
  rep = segment_scans.main(["--scans", str(tmp_path / "velodyne" / "*.bin"), "-m", "squeezesegv2", "-n",
                            "squeezesegv2kitti", "--random_init", "--batch", "2", "--output_dir", str(out),
                            "--confidence", "--temperature", "2", "--labels", str(tmp_path / "labels" / "*.label")])
  text = capsys.readouterr().out
  assert text.index("MIoU:") < text.index("RELIABILITY") and "points" in text
  mc, model = load_model_config("squeezesegv2", "squeezesegv2kitti")     # the CLI's model: same seeded init
  ev = ScanEvaluator(model, 3.0, -25.0, knn=KNN(), calibration=Calibration(temperature=2.0))
  loader = ScanBatchLoader("kitti")
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2], labs[lo:lo + 2])
    res = ev.update(data)
    pc = np.split(res["point_confidence"].cpu().numpy(), np.cumsum(data["sizes"])[:-1])
    for f, c in zip(files[lo:lo + 2], pc):
      got = np.fromfile(str(out / (os.path.splitext(os.path.basename(f))[0] + ".conf")), dtype=np.float32)
      assert got.size == c.size and np.array_equal(got, c)
  assert np.array_equal(ev.finish()["calibration"]["reliability"]["bin_count"],
                        rep["calibration"]["reliability"]["bin_count"])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_calibration_equals_single_gpu():
  cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
         "127.0.0.1", "--master-port", "29519", os.path.join(ROOT, "tests", "multi_gpu_calibration_worker.py")]
  r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
  rep = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
  assert rep["ok"] and rep["world"] == 2
