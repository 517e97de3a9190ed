"""MC dropout on the GPU (pcls_net_dropout / pcls_net_set_dropout, pcls_mc_accumulate / pcls_mc_finalize,
mc_dropout.forward_mc and its pipeline hooks): the dropout sites against the bit-exact numpy oracle
(oracle/mc_dropout.py), the merge kernels against numpy, the whole MC forward against float64, and the independence of
the results from how the work is split."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import mc_dropout as O
from oracle import nn as ONN
from tests.util import synth_range_images

pytestmark = pytest.mark.gpu

PREC = {"f16": 0, "bf16": 1}


def _lib():
  from pclsegmentation_b200 import _lib
  return _lib


def _model(name, cfg, H, W, seed=1):
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map[cfg]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = H, W
  model = model_map[name](mc)
  model.randomize_batch_norm(seed)
  return mc, model


def _mc_pass(model, net, raw, seed, frame_base, n_pass):
  """One stochastic forward of the MC net handle ``net`` on raw frames -> (probs, preds) CUDA tensors."""
  lib = _lib()
  mc = model.mc
  B, H, W, C = raw.shape
  probs = torch.empty((B, H, W, mc.NUM_CLASS), dtype=torch.float32, device="cuda")
  preds = torch.empty((B, H, W), dtype=torch.int32, device="cuda")
  s = torch.cuda.current_stream().cuda_stream
  mean = (ctypes.c_double * 5)(*np.asarray(mc.INPUT_MEAN, np.float64).reshape(-1)[:5])
  std = (ctypes.c_double * 5)(*np.asarray(mc.INPUT_STD, np.float64).reshape(-1)[:5])
  lib.check(lib.load().pcls_net_set_dropout(net, seed, frame_base, n_pass, s), "pcls_net_set_dropout")
  lib.check(lib.load().pcls_net_forward(net, raw.data_ptr(), C, None, mean, std, B, None, probs.data_ptr(),
                                        preds.data_ptr(), s), "pcls_net_forward")
  return probs, preds


SITE_CASES = [("squeezesegv2", "squeezesegv2kitti", 32, 256, 0, "fire13")] + \
             [("darknet21", "darknet21", 32, 256, k, "enc%d" % (k + 1)) for k in range(5)] + \
             [("darknet21", "darknet21", 32, 256, 5, "dec1")]


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("micro", [0, 2])
@pytest.mark.parametrize("name,cfg,H,W,site,tap", SITE_CASES)
def test_every_site_bit_exact(name, cfg, H, W, site, tap, prec, micro):
  """The MC net's tensor at a site == oracle.dropout_bits of the default net's tensor at that point (all other sites at
  rate 0, which leaves a tensor bit-for-bit unchanged), for two (seed, frame_base, pass) triples."""
  mc, model = _model(name, cfg, H, W)
  model.precision = PREC[prec]
  model.set_option("keep_tensors", 1)
  if micro:
    model.set_option("micro_batch", micro)
  B = 3
  last = B - ((B - 1) // micro) * micro if micro else B     # frames of the last pass (what the arena holds)
  first = B - last
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(site), B, H, W, channels=6)).cuda()
  model.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD)
  ref = model.read_tap(tap, last).cpu().numpy()
  n_sites = len(model._graph.dropout_sites)
  rates = [0.0] * n_sites
  rates[site] = 0.3
  net = model.mc_net(rates, B)
  for seed, fb, pss in ((0, 0, 0), ((1 << 64) - 3, (1 << 32) + 5, 65535)):
    _mc_pass(model, net, raw, seed, fb, pss)
    got = model.read_tap(tap, last, net=net).cpu().numpy()
    want = O.dropout_bits(O.from_f32(ref, prec), prec, seed, fb + first, pss, site, 0.3)
    assert np.array_equal(O.from_f32(got, prec), want), (seed, fb, pss)
    assert 0.6 < (want != 0).mean() < 0.8 or (ref == 0).mean() > 0.2
  model._release()


def _mc_vs_plain(model, mc, raw, T):
  from pclsegmentation_b200.mc_dropout import MCDropout, forward_mc
  from pclsegmentation_b200.calibration import confidence, raw_mask
  plain = model.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD)
  got = forward_mc(model, raw, MCDropout(passes=T, seed=7, rate=0.0), want_probabilities=True)
  c = confidence(mc.NUM_CLASS, probs=plain["probabilities"], mask=raw_mask(raw, mc), want_entropy=True)
  return plain, got, c


@pytest.mark.parametrize("name,cfg,H,W", [("squeezesegv2", "squeezesegv2kitti", 64, 512),
                                          ("darknet21", "darknet21", 32, 256)])
def test_rate_zero_equals_the_plain_forward(name, cfg, H, W):
  """At rate 0, T = 1 and 2 give the plain forward's probabilities and predictions bit for bit, MI exactly 0 and H ==
  pcls_confidence's entropy; T = 4 sums four equal float32 values in order (3p rounds), so it is only within 4 ulp."""
  mc, model = _model(name, cfg, H, W)
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(3), 2, H, W, channels=6)).cuda()
  for T in (1, 2):
    plain, got, c = _mc_vs_plain(model, mc, raw, T)
    assert torch.equal(got["probabilities"], plain["probabilities"])
    assert torch.equal(got["predictions"], plain["predictions"])
    assert (got["mutual_information"] == 0).all()
    assert torch.equal(got["entropy"], c["entropy"])
    assert torch.equal(got["confidence"], c["confidence"])
  plain, got, c = _mc_vs_plain(model, mc, raw, 4)
  assert (got["probabilities"] - plain["probabilities"]).abs().max().item() <= 1e-6
  assert (got["mutual_information"] >= 0).all() and got["mutual_information"].max().item() < 1e-5
  model._release()


@pytest.mark.parametrize("name,cfg,H,W,B", [("squeezesegv2", "squeezesegv2kitti", 32, 256, 2),
                                            ("darknet21", "darknet21", 32, 240, 2)])
def test_whole_mc_forward_against_float64(name, cfg, H, W, B):
  """Rate 0.5, T = 4: every pass's probabilities against oracle.nn with the same masks in float64, within the logits
  tolerance of test_gpu_nets (probabilities are 1-Lipschitz in the logits), and the finalize of those passes."""
  from tests.test_gpu_nets import LOGIT_TOL
  mc, model = _model(name, cfg, H, W)
  raw = synth_range_images(np.random.default_rng(11), B, H, W, channels=6)
  lidar = np.stack([ONN.input_stage(r, mc.INPUT_MEAN, mc.INPUT_STD, mc.CLASSES.index("None"))[0] for r in raw])
  mask = lidar[..., 5] > 0
  arch = "squeezesegv2" if name.startswith("squeeze") else "darknet"
  nl = 21 if name == "darknet21" else 53
  params = model.get_weights_dict()
  net = model.mc_net(0.5, B)
  rawd = torch.from_numpy(raw).cuda()
  for t in range(4):
    probs, _ = _mc_pass(model, net, rawd, 9, 100, t)
    drop = lambda k, x: O.apply_dropout(x, 9, 100, t, k, 0.5)
    lg, pr, _ = O.forward(arch, params, lidar, mask, mc.CLASSES.index("None"), drop, num_layers=nl,
                          output_stride=getattr(mc, "OUTPUT_STRIDE", 16))
    scale = max(1.0, float(np.abs(lg).max()) / 4.0)
    err = np.abs(probs.cpu().numpy() - pr).max()
    assert err <= 2 * LOGIT_TOL * scale, (t, err)
  model._release()


@pytest.mark.parametrize("nc", [11, 20])
def test_accumulate_finalize_against_numpy(nc):
  """Mean and predictions exact (float32 sums in pass order, planted ties), H / MI within 8 float32 ulp of 1 (numpy's
  float32 log may differ from logf in the last bit), masked pixels zero."""
  from pclsegmentation_b200.mc_dropout import accumulate, finalize
  rng = np.random.default_rng(nc)
  n, T = 5000, 5
  ps = []
  for t in range(T):
    z = rng.normal(0, 2, (n, nc)).astype(np.float32)
    p = np.exp(z - z.max(axis=1, keepdims=True))
    p = (p / p.sum(axis=1, keepdims=True)).astype(np.float32)
    p[:50] = np.float32(1.0 / nc)                               # planted ties
    p[50:60, 1:] = 0
    p[50:60, 0] = 1
    ps.append(p)
  mask = (rng.random(n) > 0.1).astype(np.uint8)
  acc_p = torch.empty((n, nc), dtype=torch.float32, device="cuda")
  acc_h = torch.empty(n, dtype=torch.float64, device="cuda")
  for t, p in enumerate(ps):
    accumulate(torch.from_numpy(p).cuda(), t, acc_p, acc_h, nc)
  want_a, want_h = O.accumulate(ps)
  assert np.array_equal(acc_p.cpu().numpy(), want_a)
  assert np.abs(acc_h.cpu().numpy() - want_h).max() <= T * 8 * 2 ** -24
  got = finalize(acc_p, acc_h, torch.from_numpy(mask).cuda(), nc, nc - 1, T)
  want = O.finalize(want_a, acc_h.cpu().numpy(), mask, T, nc - 1)
  assert np.array_equal(got["probabilities"].cpu().numpy(), want["probabilities"])
  assert np.array_equal(got["predictions"].cpu().numpy(), want["predictions"])
  assert np.array_equal(got["confidence"].cpu().numpy(), want["confidence"])
  for k in ("entropy", "mutual_information"):
    assert np.abs(got[k].cpu().numpy() - want[k]).max() <= 8 * 2 ** -24, k
    assert (got[k].cpu().numpy()[mask == 0] == 0).all()
  assert (got["predictions"].cpu().numpy()[:50][mask[:50] != 0] == 0).all()


def _mc_run(model, mc, raw, **opts):
  from pclsegmentation_b200.mc_dropout import MCDropout, forward_mc
  m = MCDropout(passes=3, seed=42, rate=0.2)
  outs = []
  for part in opts.get("split", [raw]):
    outs.append(forward_mc(model, part, m, want_probabilities=True))
  return {k: torch.cat([o[k] for o in outs]) for k in outs[0]}


def test_independent_of_how_the_work_is_split():
  """One call with B = 4 == two calls with B = 2 (next_frame carries on) == micro_batch 1 == plain launches."""
  mc, model = _model("squeezesegv2", "squeezesegv2kitti", 32, 512)
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(5), 4, 32, 512, channels=6)).cuda()
  a = _mc_run(model, mc, raw)
  b = _mc_run(model, mc, raw, split=[raw[:2].contiguous(), raw[2:].contiguous()])
  model.set_option("micro_batch", 1)
  c = _mc_run(model, mc, raw)
  model.set_option("micro_batch", 0)
  model.set_option("use_graph", 0)
  d = _mc_run(model, mc, raw)
  for other in (b, c, d):
    for k in a:
      assert torch.equal(a[k], other[k]), k
  assert (a["mutual_information"] > 0).any()
  model._release()


def test_graph_replay_reads_the_state():
  """The captured graph is replayed with the state written before it: pass 0 and pass 1 differ, the same state twice
  gives the same bits."""
  mc, model = _model("squeezesegv2", "squeezesegv2kitti", 32, 512)
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(6), 2, 32, 512, channels=6)).cuda()
  net = model.mc_net(0.3, 2)
  p0 = _mc_pass(model, net, raw, 1, 0, 0)[0].clone()
  p1 = _mc_pass(model, net, raw, 1, 0, 1)[0].clone()
  p0b = _mc_pass(model, net, raw, 1, 0, 0)[0].clone()
  p2 = _mc_pass(model, net, raw, 1, 2, 0)[0].clone()
  assert not torch.equal(p0, p1) and not torch.equal(p0, p2)
  assert torch.equal(p0, p0b)
  model._release()


def test_default_net_is_untouched():
  """After an MC net has been built and run, the default forward gives a fresh model's bits, with the same op count
  and launches per forward."""
  from pclsegmentation_b200.mc_dropout import MCDropout, forward_mc
  lib = _lib().load()
  mc, model = _model("squeezesegv2", "squeezesegv2kitti", 64, 512)
  mc2, fresh = _model("squeezesegv2", "squeezesegv2kitti", 64, 512)
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(8), 2, 64, 512, channels=6)).cuda()
  want = fresh.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD)
  forward_mc(model, raw, MCDropout(passes=2, rate=0.1))
  got = model.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD)
  assert torch.equal(got["probabilities"], want["probabilities"])
  assert torch.equal(got["predictions"], want["predictions"])
  assert lib.pcls_net_num_ops(model._net) == lib.pcls_net_num_ops(fresh._net)
  assert lib.pcls_net_launches_per_forward(model._net) == lib.pcls_net_launches_per_forward(fresh._net)
  mcn = model.mc_net(0.1, 2)
  assert lib.pcls_net_num_ops(mcn) == lib.pcls_net_num_ops(fresh._net) + 1
  names = []
  for i in range(lib.pcls_net_num_ops(mcn)):
    buf = ctypes.create_string_buffer(64)
    fam, fl, by = ctypes.c_int(), ctypes.c_int64(), ctypes.c_int64()
    assert lib.pcls_net_op_info(mcn, i, buf, ctypes.byref(fam), ctypes.byref(fl), ctypes.byref(by)) == 0
    names.append((buf.value.decode(), by.value))
  assert ("dropout_s0_c64_w512", 64 * 512 * 64 * 4) in names
  model._release()
  fresh._release()


def test_net_dropout_refusals():
  """pcls_net_dropout refuses the input, logits, padded tensors, duplicate sites, bad rates, finalized nets."""
  import ctypes as C
  lib = _lib().load()
  h = C.c_void_p()
  assert lib.pcls_net_create(C.byref(h), 4, 16, 0, 1) == 0
  t1 = lib.pcls_net_tensor(h, 16, 16, 0)
  assert lib.pcls_net_dropout(h, t1, 0, 0.1) == -1 and b"not written" in lib.pcls_last_error()
  assert lib.pcls_net_dropout(h, 0, 0, 0.1) == -1 and b"network input" in lib.pcls_last_error()
  k = (C.c_float * (6 * 16))(*([0.1] * 96))
  d = _lib().ConvDesc(kind=0, kh=1, kw=1, stride_w=1, cin=6, cout=16, h_kernel=k, bn_eps=1e-3, act=1, in_tensor=0,
                      out_tensor=t1, out_channel_offset=0, residual0=-1, residual1=-1, out_is_logits=0)
  assert lib.pcls_net_conv(h, C.byref(d)) == 0
  for site, rate, msg in ((0, -0.1, b"rate"), (0, 1.0, b"rate"), (0, float("nan"), b"rate"), (65536, 0.1, b"site")):
    assert lib.pcls_net_dropout(h, t1, site, rate) == -1 and msg in lib.pcls_last_error(), (site, rate)
  assert lib.pcls_net_dropout(h, t1, 0, 0.1) == 0
  assert lib.pcls_net_dropout(h, t1, 0, 0.1) == -1 and b"twice" in lib.pcls_last_error()
  assert lib.pcls_net_set_dropout(h, 0, 0, 0, None) == -1 and b"finalized" in lib.pcls_last_error()
  lib.pcls_net_destroy(h)


def test_evaluator_and_scan_segmenter_at_rate_zero():
  """At rate 0 (T = 2) the Evaluator's confusion matrix and the ScanSegmenter's predictions equal the plain runs; the
  point MI gather is exact; MC + TTA and MC + temperature are refused."""
  from pclsegmentation_b200.calibration import Calibration
  from pclsegmentation_b200.mc_dropout import MCDropout
  from pclsegmentation_b200.pipeline import Evaluator, ScanSegmenter
  from pclsegmentation_b200.tta import TTA
  from tests.util import synth_scan
  mc, model = _model("squeezesegv2", "squeezesegv2kitti", 64, 512)
  raw = synth_range_images(np.random.default_rng(9), 3, 64, 512, channels=6, num_classes=mc.NUM_CLASS)
  plain, mcd = Evaluator(model), Evaluator(model, mc_dropout=MCDropout(passes=2, rate=0.0))
  plain.update(raw)
  mcd.update(raw)
  a, b = plain.finish(), mcd.finish()
  assert np.array_equal(a["confusion_matrix"], b["confusion_matrix"])
  u = b["mc_dropout"]["uncertainty"]
  assert u["count"] > 0 and 0.0 <= u["auroc_entropy"] <= 1.0
  assert (u["mi_count"][1:] == 0).all()                          # MI is exactly 0 at rate 0, T = 2
  with pytest.raises(ValueError):
    Evaluator(model, tta=TTA(), mc_dropout=MCDropout())
  with pytest.raises(ValueError):
    Evaluator(model, calibration=Calibration(temperature=2.0), mc_dropout=MCDropout())
  seg = ScanSegmenter(model)
  rng = np.random.default_rng(2)
  scans = [synth_scan(rng, 20000) for _ in range(2)]
  pts = torch.from_numpy(np.concatenate(scans)[:, :4].astype(np.float32)).cuda()
  off = torch.tensor([0, len(scans[0]), len(scans[0]) + len(scans[1])], dtype=torch.int64).cuda()
  r0 = seg.segment_device(pts, off, want_point_labels=True)
  r1 = seg.segment_device(pts, off, want_point_labels=True, mc_dropout=MCDropout(passes=2, rate=0.0, seed=3))
  assert torch.equal(r0["predictions"], r1["predictions"]) and torch.equal(r0["point_labels"], r1["point_labels"])
  r2 = seg.segment_device(pts, off, want_point_labels=True, mc_dropout=MCDropout(passes=2, rate=0.5, seed=3),
                          want_image=True, want_probabilities=True)
  mi = r2["mutual_information"].cpu().numpy()
  proj = seg.projector.project(pts, off, want_point_outputs=True)
  px, py = proj["proj_x"].cpu().numpy(), proj["proj_y"].cpu().numpy()
  sizes = [len(s) for s in scans]
  b_of = np.repeat(np.arange(2), sizes)
  want = np.where(px >= 0, mi[b_of, np.maximum(py, 0), np.maximum(px, 0)], 0).astype(np.float32)
  assert np.array_equal(r2["point_mi"].cpu().numpy(), want)
  assert (want > 0).any()
  # the point confidence is the MC mean's probability of the point's own label (as with confidence=1)
  pr, lab = r2["probabilities"].cpu().numpy(), r2["point_labels"].cpu().numpy()
  want_c = np.where(px >= 0, pr[b_of, np.maximum(py, 0), np.maximum(px, 0), np.clip(lab, 0, mc.NUM_CLASS - 1)], 0)
  assert np.array_equal(r2["point_confidence"].cpu().numpy(), want_c.astype(np.float32))
  r3 = seg.segment_device(pts, off, want_point_labels=True, mc_dropout=MCDropout(passes=2, rate=0.5, seed=3),
                          confidence=1.0)
  assert torch.equal(r3["point_confidence"], r2["point_confidence"]) and "probabilities" not in r3
  with pytest.raises(ValueError):
    seg.segment_device(pts, off, tta=TTA(), mc_dropout=MCDropout())
  model._release()


@pytest.fixture(scope="module")
def golden(golden_dir):
  import os
  with np.load(os.path.join(golden_dir, "nn_sample_dataset.npz")) as f:
    return {k: f[k] for k in f.files}


def test_inference_and_eval_cli_with_mc_dropout(tmp_path, golden, capsys):
  """inference writes unc_<name>.npy ([H,W,2] = H, MI) and the MC confidence; eval prints the MC report after the mIoU
  report with the MC predictions' confusion matrix; MC + TTA and MC + temperature are refused."""
  import os
  from oracle import confusion as C
  from pclsegmentation_b200 import eval as ev
  from pclsegmentation_b200 import inference
  from pclsegmentation_b200.mc_dropout import MCDropout, forward_mc
  from tests.test_gpu_tta import _sample_model
  mc, model, wpath = _sample_model(tmp_path)
  d = tmp_path / "data" / "val"
  d.mkdir(parents=True)
  for n, f in zip(golden["names"], golden["frames"]):
    np.save(str(d / str(n)), f.astype(np.float64))
  frames = torch.from_numpy(golden["frames"].astype(np.float32)).cuda()
  mcd = MCDropout(passes=3, seed=5, rate=0.3)
  want = {}
  for lo in range(0, frames.shape[0], 2):      # the CLI's batches of 2, next_frame carried on
    r = forward_mc(model, frames[lo:lo + 2].contiguous(), mcd)
    for k, v in r.items():
      want.setdefault(k, []).append(v.cpu().numpy())
  want = {k: np.concatenate(v) for k, v in want.items()}
  outdir = tmp_path / "out"
  mcargs = ["--mc_dropout", "3", "--mc_seed", "5", "--mc_rate", "0.3"]
  inference.main(["-d", str(d / "*.npy"), "-m", "squeezesegv2", "-n", "squeezesegv2", "-t", str(outdir), "-p", wpath,
                  "-b", "2", "--no_plots", "--confidence"] + mcargs)
  for i, n in enumerate(golden["names"]):
    stem = os.path.splitext(str(n))[0]
    assert np.array_equal(np.load(str(outdir / ("pred_" + stem + ".npy"))), want["predictions"][i])
    unc = np.load(str(outdir / ("unc_" + stem + ".npy")))
    assert unc.shape == frames.shape[1:3] + (2,) and unc.dtype == np.float32
    assert np.array_equal(unc[..., 0], want["entropy"][i]) and np.array_equal(unc[..., 1], want["mutual_information"][i])
    assert np.array_equal(np.load(str(outdir / ("conf_" + stem + ".npy"))), want["confidence"][i])
  rep = ev.main(["-d", str(tmp_path / "data"), "-i", "val", "-m", "squeezesegv2", "-n", "squeezesegv2", "-p", wpath,
                 "-b", "2"] + mcargs)
  out = capsys.readouterr().out
  assert out.index("MIoU:") < out.index("MC DROPOUT T = 3") < out.index("AUROC(MI):")
  cm = C.confusion_matrix(golden["label"].astype(np.int32), want["predictions"], mc.NUM_CLASS)
  assert np.array_equal(rep["confusion_matrix"], cm)
  with pytest.raises(SystemExit):
    inference.main(["-d", str(d / "*.npy"), "-m", "squeezesegv2", "-n", "squeezesegv2", "-t", str(outdir), "-p", wpath,
                    "--no_plots", "--tta"] + mcargs)
  with pytest.raises(SystemExit):
    ev.main(["-d", str(tmp_path / "data"), "-i", "val", "-m", "squeezesegv2", "-n", "squeezesegv2", "-p", wpath,
             "--calibration", "--temperature", "1.5"] + mcargs)


def test_segment_scans_cli_and_scan_evaluator_with_mc_dropout(tmp_path, capsys):
  """segment_scans writes <name>.unc (the points' MI) and, with --labels, the point-wise MC report; ScanEvaluator at
  rate 0 gives the plain confusion matrix."""
  import os
  from pclsegmentation_b200 import segment_scans
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader
  from pclsegmentation_b200.mc_dropout import MCDropout
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  from pclsegmentation_b200.utils.args_loader import load_model_config
  from tests.test_gpu_tta import _write_kitti
  rng = np.random.default_rng(12)
  scan_dir, lab_dir = _write_kitti(tmp_path, rng, [8000, 6000, 7000])
  out = tmp_path / "pred"
  args = ["--scans", str(scan_dir / "*.bin"), "-m", "squeezesegv2", "-n", "squeezesegv2kitti", "--random_init",
          "--batch", "2", "--output_dir", str(out), "--mc_dropout", "2", "--mc_rate", "0.4"]
  rep_cli = segment_scans.main(args + ["--labels", str(lab_dir / "*.label")])
  assert "AUROC(H):" in capsys.readouterr().out
  mc, model = load_model_config("squeezesegv2", "squeezesegv2kitti")
  ev = ScanEvaluator(model, 3.0, -25.0, knn=KNN(), mc_dropout=MCDropout(passes=2, rate=0.4))
  loader = ScanBatchLoader("kitti")
  files = sorted(str(p) for p in scan_dir.iterdir())
  labs = sorted(str(p) for p in lab_dir.iterdir())
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2], labs[lo:lo + 2])
    res = ev.update(data)
    for f, u in zip(files[lo:lo + 2], np.split(res["point_mi"].cpu().numpy(), np.cumsum(data["sizes"])[:-1])):
      got = np.fromfile(str(out / (os.path.splitext(os.path.basename(f))[0] + ".unc")), dtype=np.float32)
      assert np.array_equal(got, u)
  rep = ev.finish()
  assert np.array_equal(rep_cli["confusion_matrix"], rep["confusion_matrix"])
  assert np.array_equal(rep_cli["mc_dropout"]["uncertainty"]["mi_count"], rep["mc_dropout"]["uncertainty"]["mi_count"])
  plain = ScanEvaluator(model, 3.0, -25.0, knn=KNN())
  zero = ScanEvaluator(model, 3.0, -25.0, knn=KNN(), mc_dropout=MCDropout(passes=2, rate=0.0))
  data = loader.load(files[:2], labs[:2])
  plain.update(data)
  zero.update(data)
  assert np.array_equal(plain.finish()["confusion_matrix"], zero.finish()["confusion_matrix"])


def test_shards_with_global_frame_ids_equal_one_run():
  """What a sharded eval does, on one GPU: each shard's Evaluator starts its frame counter at the shard's first global
  frame index (eval.py under torchrun); the shards' confusion matrices and integer uncertainty / reliability bins sum
  to exactly the single run's, whatever the batching."""
  from pclsegmentation_b200.mc_dropout import MCDropout
  from pclsegmentation_b200.pipeline import Evaluator
  from pclsegmentation_b200.sharding import shard_range
  mc, model = _model("squeezesegv2", "squeezesegv2nuscenes", 32, 256)
  frames = synth_range_images(np.random.default_rng(79), 13, 32, 256, valid_rate=0.6, num_classes=11)
  solo = Evaluator(model, mc_dropout=MCDropout(passes=3, seed=17, rate=0.4))
  for i in range(0, 13, 5):
    solo.update(frames[i:i + 5])
  ref = solo.finish()
  keys = ("entropy_count", "entropy_correct", "mi_count", "mi_correct")
  cm, bins, rel = 0, {k: 0 for k in keys}, 0
  for rank in range(3):
    lo, hi = shard_range(13, rank, 3)
    mcd = MCDropout(passes=3, seed=17, rate=0.4)
    mcd.next_frame = lo
    ev = Evaluator(model, mc_dropout=mcd)
    for i in range(lo, hi, 2):
      ev.update(frames[i:min(i + 2, hi)])
    rep = ev.finish()
    cm = cm + rep["confusion_matrix"]
    rel = rel + rep["mc_dropout"]["reliability"]["bin_count"]
    for k in keys:
      bins[k] = bins[k] + rep["mc_dropout"]["uncertainty"][k]
  assert np.array_equal(cm, ref["confusion_matrix"])
  assert np.array_equal(rel, ref["mc_dropout"]["reliability"]["bin_count"])
  for k in keys:
    assert np.array_equal(bins[k], ref["mc_dropout"]["uncertainty"][k]), k
  assert (ref["mc_dropout"]["uncertainty"]["mi_count"][1:] > 0).any()
  model._release()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_mc_eval_equals_single_gpu():
  import json
  import os
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
         "127.0.0.1", "--master-port", "29523", os.path.join(root, "tests", "multi_gpu_mc_dropout_worker.py")]
  r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
  rep = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
  assert rep["ok"] and rep["world"] == 2
