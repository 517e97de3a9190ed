"""Test-time augmentation on the GPU (pcls_tta_views, pcls_tta_merge, tta.forward_tta and its pipelines / CLIs):
every comparison is `==` on bits against the numpy oracle (oracle/tta.py) or against the plain path."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import confusion as C
from oracle import point_labels as PL
from oracle import tta as O
from tests.util import synth_range_images, synth_scan

pytestmark = pytest.mark.gpu

G = 64                  # guard band, elements
GUARD16, GUARD8 = 0x5A5A, 0xA5
SENT16, SENT8 = 0x7C01, 0xCD    # sentinel prefill (an fp16 NaN / a mask byte that is neither 0 nor 1)
PREC = {"f16": 0, "bf16": 1}


def _lib():
  from pclsegmentation_b200 import _lib
  return _lib


def _arr(t, v):
  return (t * len(v))(*[x.item() if hasattr(x, "item") else x for x in v])


def _views_arrays(views, W):
  flip = [f for f, _ in views]
  shift = [s for _, s in views]
  cs = [O.rotation(s, W) for s in shift]
  return (_arr(ctypes.c_int, flip), _arr(ctypes.c_int, shift), _arr(ctypes.c_double, [c for c, _ in cs]),
          _arr(ctypes.c_double, [s for _, s in cs]))


def device_views(raw, mean, std, views, prec):
  """pcls_tta_views into guard-banded, sentinel-prefilled buffers; checks the bands and returns (input uint16, mask)."""
  lib = _lib()
  B, H, W, C = raw.shape
  n = len(views) * B * H * W
  ibuf = torch.full((n * 8 + 2 * G,), SENT16, dtype=torch.int32, device="cuda").to(torch.int16)
  ibuf[:G] = GUARD16
  ibuf[G + n * 8:] = GUARD16
  mbuf = torch.full((n + 2 * G,), SENT8, dtype=torch.uint8, device="cuda")
  mbuf[:G] = GUARD8
  mbuf[G + n:] = GUARD8
  f, s, c, sn = _views_arrays(views, W)
  lib.check(lib.load().pcls_tta_views(raw.data_ptr(), C, B, H, W, _arr(ctypes.c_double, mean), _arr(ctypes.c_double, std),
                                      len(views), f, s, c, sn, PREC[prec], ibuf[G:].data_ptr(), mbuf[G:].data_ptr(),
                                      torch.cuda.current_stream().cuda_stream), "pcls_tta_views")
  ih = ibuf.cpu().numpy().view(np.uint16)
  mh = mbuf.cpu().numpy()
  assert (ih[:G] == GUARD16).all() and (ih[G + n * 8:] == GUARD16).all(), "input guard band written"
  assert (mh[:G] == GUARD8).all() and (mh[G + n:] == GUARD8).all(), "mask guard band written"
  assert not (mh[G:G + n] == SENT8).any(), "a mask byte was not written"
  return ih[G:G + n * 8].reshape(len(views) * B, H, W, 8), mh[G:G + n].reshape(len(views) * B, H, W)


def hard_raw(rng, B, H, W, channels):
  """Range images with signed values, empty pixels of every kind (range 0, negative, NaN), signed zeros and large
  magnitudes (past the fp16 range)."""
  raw = synth_range_images(rng, B, H, W, channels=channels)
  n = raw[..., 0].size
  flat = raw.reshape(n, channels)
  idx = rng.choice(n, n // 10, replace=False)
  flat[idx[:n // 40], :2] *= -1e6                          # |x|, |y| up to 8e7: inf in fp16, finite in bf16
  flat[idx[n // 40:n // 20], 0] = -0.0
  flat[idx[n // 40:n // 20], 1] = -0.0
  flat[idx[n // 20:n // 15], 4] = -3.0                     # negative range: empty, with non-zero x, y, z
  flat[idx[n // 15:n // 12], 4] = np.nan
  flat[idx[n // 12:], :4] = rng.normal(0, 1e3, (idx.size - n // 12, 4))
  return raw


VIEW_SETS = lambda W: [
  [(0, 0)], [(1, 0)], [(0, 1)], [(1, W - 1)], [(0, W // 4)],
  [(0, 0), (1, 0)],
  [(0, 0), (0, W // 2), (1, 0), (1, W // 2)],
  [(1, 3), (0, 0), (0, W // 4)],
  [(0, 5), (1, 5), (0, 0), (1, W // 2), (0, W - 1)],
  [(0, 0), (0, 1), (0, W // 4), (0, W // 2), (1, 0), (1, W - 1), (1, 7), (0, 13)][:6],
  [(0, 0), (0, 1), (0, W // 4), (0, W // 2), (1, 0), (1, W - 1), (1, 7), (0, 13)][:7],
  [(0, 0), (0, 1), (0, W // 4), (0, W // 2), (1, 0), (1, W - 1), (1, 7), (0, 13)],
]


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("channels", [5, 6])
@pytest.mark.parametrize("shape", [(3, 4, 64), (2, 5, 50), (2, 64, 2048)])
def test_views_equal_oracle(prec, channels, shape):
  B, H, W = shape
  rng = np.random.default_rng(B * 1000 + W + channels)
  raw = hard_raw(rng, B, H, W, channels)
  d = torch.from_numpy(raw).cuda()
  mean = [10.5, -0.25, -1.1, 0.21, 12.0]
  std = [11.7, 9.3, 0.8, 0.14, 12.3]
  for views in VIEW_SETS(W):
    got, gm = device_views(d, mean, std, views, prec)
    want, wm = O.views_input(raw, mean, std, views, prec)
    assert np.array_equal(gm, wm), views
    bad = np.argwhere(got != want)
    assert bad.size == 0, (views, bad[:5], got[tuple(bad[0])], want[tuple(bad[0])])


@pytest.mark.parametrize("prec", ["f16", "bf16"])
def test_view_zero_is_the_net_input(prec):
  """View (0, 0) is bit-identical to the tensor 0 the forward makes of raw input: the forward over it (staged) gives
  the raw forward's bits."""
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map["squeezesegv2kitti"]()
  mc.AZIMUTH_LEVEL = 256
  model = model_map["squeezesegv2"](mc)
  model.precision = PREC[prec]
  model.randomize_batch_norm(4)
  raw = hard_raw(np.random.default_rng(9), 3, 64, 256, 5)
  raw[..., :2] = np.clip(raw[..., :2], -100, 100)
  d = torch.from_numpy(raw).cuda()
  want = model.forward_device(d, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD, want_logits=True)
  inp, msk, frames = model.input_buffers(3)
  f, s, c, sn = _views_arrays([(0, 0)], 256)
  lib = _lib()
  mean = _arr(ctypes.c_double, np.asarray(mc.INPUT_MEAN, np.float64).reshape(-1))
  std = _arr(ctypes.c_double, np.asarray(mc.INPUT_STD, np.float64).reshape(-1))
  lib.check(lib.load().pcls_tta_views(d.data_ptr(), 5, 3, 64, 256, mean, std, 1, f, s, c, sn, model.precision, inp, msk,
                                      torch.cuda.current_stream().cuda_stream), "pcls_tta_views")
  got = model.forward_staged(3, want_logits=True)
  for k in ("logits", "probabilities", "predictions"):
    assert torch.equal(got[k], want[k]), k
  model._release()


def planted_probs(rng, n, H, W, nc):
  """Probabilities on a 1/8 grid (sums and means of several views tie exactly) and a few NaN rows."""
  p = (rng.integers(0, 9, (n, H, W, nc)) / 8.0).astype(np.float32)
  p[:, 0, 0, :] = 0.25                                     # all classes tie
  p[rng.random((n, H, W)) < 0.01] = np.float32(np.nan)
  return p


@pytest.mark.parametrize("nc", [11, 20, 32])
def test_merge_equals_oracle(nc):
  lib = _lib()
  rng = np.random.default_rng(nc)
  for (B, H, W) in ((3, 5, 70), (2, 4, 64)):
    for T in range(1, 9):
      views = [(0, 0), (1, W - 1), (0, 3), (1, 0), (0, W // 2), (1, 7), (0, W - 1), (1, W // 4)][:T]
      if T % 2 == 0:
        views = views[::-1]                                # view 0 not the identity
      probs = planted_probs(rng, T * B, H, W, nc)
      mask = (rng.random((T * B, H, W)) < 0.8).astype(np.uint8)
      none = nc - 1 - T % 3
      want_p, want_y = O.merge(probs, mask, views, none)
      assert (want_y == none).any() and (want_y != none).any()
      f, s, _, _ = _views_arrays(views, W)
      dp, dm = torch.from_numpy(probs).cuda(), torch.from_numpy(mask).cuda()
      n = B * H * W
      for with_probs in (True, False):
        ybuf = torch.full((n + 2 * G,), -7, dtype=torch.int32, device="cuda")
        ybuf[:G] = 0x5A5A5A5A
        ybuf[G + n:] = 0x5A5A5A5A
        pbuf = torch.full((n * nc + 2 * G,), -3.0, dtype=torch.float32, device="cuda")
        pbuf[:G] = 1e30
        pbuf[G + n * nc:] = 1e30
        lib.check(lib.load().pcls_tta_merge(dp.data_ptr(), dm.data_ptr(), B, H, W, nc, none, T, f, s,
                                            pbuf[G:].data_ptr() if with_probs else None, ybuf[G:].data_ptr(),
                                            torch.cuda.current_stream().cuda_stream), "pcls_tta_merge")
        y, p = ybuf.cpu().numpy(), pbuf.cpu().numpy()
        assert (y[:G] == 0x5A5A5A5A).all() and (y[G + n:] == 0x5A5A5A5A).all()
        assert (p[:G] == np.float32(1e30)).all() and (p[G + n * nc:] == np.float32(1e30)).all()
        assert np.array_equal(y[G:G + n].reshape(B, H, W), want_y), (T, W, with_probs)
        if with_probs:
          got = p[G:G + n * nc].reshape(B, H, W, nc)
          nan = np.isnan(want_p)                           # (NaN payloads differ between the device and numpy)
          assert nan.any() and np.array_equal(np.isnan(got), nan)
          assert np.array_equal(got[~nan].view(np.uint32), want_p[~nan].view(np.uint32)), (T, W)
        else:
          assert (p[G:G + n * nc] == -3.0).all(), "merged probabilities written without out_probs"


def _kitti_model(W=2048, seed=1, name="squeezesegv2", cfg="squeezesegv2kitti"):
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map[cfg]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = 64, W
  model = model_map[name](mc)
  model.randomize_batch_norm(seed)
  return mc, model


@pytest.mark.parametrize("name,cfg,B", [("squeezesegv2", "squeezesegv2kitti", 32), ("darknet21", "darknet21", 2)])
def test_identity_tta_equals_the_plain_forward(name, cfg, B):
  from pclsegmentation_b200.tta import TTA, forward_tta
  mc, model = _kitti_model(name=name, cfg=cfg)
  raw = torch.from_numpy(synth_range_images(np.random.default_rng(B), B, 64, 2048, channels=6)).cuda()
  want = model.forward_device(raw, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD)
  got = forward_tta(model, raw, TTA(flip=False, shifts=(0,)), want_probabilities=True)
  assert torch.equal(got["probabilities"], want["probabilities"])
  assert torch.equal(got["predictions"], want["predictions"])
  model._release()


@pytest.mark.parametrize("prec", ["f16", "bf16"])
@pytest.mark.parametrize("shifts", [(0,), (0, 1024)])
def test_forward_tta_end_to_end_at_the_benchmark_shape(prec, shifts):
  """forward_tta on 32 frames of 64 x 2048 against: the oracle's 16-bit input of every view through forward_device on
  the same model, merged in numpy.  Then once more with micro_batch set (the unstaged route)."""
  from pclsegmentation_b200.tta import TTA, forward_tta
  mc, model = _kitti_model()
  model.precision = PREC[prec]
  tta = TTA(flip=True, shifts=shifts)
  B = 32
  raw = synth_range_images(np.random.default_rng(len(shifts)), B, 64, 2048, channels=6)
  got = forward_tta(model, torch.from_numpy(raw).cuda(), tta, want_probabilities=True)
  gp, gy = got["probabilities"].cpu().numpy(), got["predictions"].cpu().numpy()
  x16, m = O.views_input(raw, mc.INPUT_MEAN, mc.INPUT_STD, tta.view_list, prec)
  dt = torch.float16 if prec == "f16" else torch.bfloat16
  ref = model.forward_device(torch.from_numpy(x16.view(np.int16)).cuda().view(dt), torch.from_numpy(m).cuda())
  want_p, want_y = O.merge(ref["probabilities"].cpu().numpy(), m, tta.view_list, mc.CLASSES.index("None"))
  del ref
  assert np.array_equal(gy, want_y)
  assert np.array_equal(gp.view(np.uint32), want_p.view(np.uint32))
  assert len(np.unique(gy)) > 3
  model.set_option("micro_batch", 24)
  assert model.input_buffers(len(tta) * B)[2] < len(tta) * B
  again = forward_tta(model, torch.from_numpy(raw).cuda(), tta, want_probabilities=True)
  assert torch.equal(again["predictions"], got["predictions"])
  assert torch.equal(again["probabilities"], got["probabilities"])
  model._release()


def test_forward_tta_rejects_normalised_or_16_bit_input():
  from pclsegmentation_b200.tta import TTA, forward_tta
  mc, model = _kitti_model(W=256)
  for bad in (torch.zeros((1, 64, 256, 8), dtype=torch.float16, device="cuda"),
              torch.zeros((1, 64, 256, 7), dtype=torch.float32, device="cuda"),
              np.zeros((1, 64, 256, 6), np.float32)):
    with pytest.raises(ValueError, match="RAW"):
      forward_tta(model, bad, TTA())


# ---- pipelines ----

@pytest.fixture(scope="module")
def small_model():
  return _kitti_model(W=512, seed=2)


@pytest.fixture(scope="module")
def scans():
  rng = np.random.default_rng(8)
  sizes = [20000, 0, 15000, 1]
  pts = [synth_scan(rng, n) for n in sizes]
  return sizes, pts


def _scan_tensors(sizes, pts):
  return (torch.from_numpy(np.concatenate(pts)).cuda(),
          torch.as_tensor(np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)).cuda())


def test_identity_tta_scan_path_equals_the_staged_path(small_model, scans):
  from pclsegmentation_b200.pipeline import KNN, Clustering, ScanSegmenter
  from pclsegmentation_b200.tta import TTA
  mc, model = small_model
  pts, offsets = _scan_tensors(*scans)
  seg = ScanSegmenter(model, 3.0, -25.0)
  kw = dict(want_point_labels=True, knn=KNN(), instances=Clustering())
  plain = seg.segment_device(pts, offsets, want_probabilities=True, **kw)      # staged resolve_net_input path
  ident = seg.segment_device(pts, offsets, want_probabilities=True, tta=TTA(flip=False), **kw)
  for k in ("predictions", "probabilities", "point_labels", "instances", "instance_counts", "proj_idx"):
    assert torch.equal(plain[k], ident[k]), k
  with pytest.raises(ValueError, match="logits"):
    seg.segment_device(pts, offsets, want_logits=True, tta=TTA())


def test_segment_device_with_tta_feeds_the_merged_predictions(small_model, scans):
  from pclsegmentation_b200.pipeline import KNN, ScanSegmenter
  from pclsegmentation_b200.tta import TTA, forward_tta
  mc, model = small_model
  sizes, _ = scans
  pts, offsets = _scan_tensors(*scans)
  seg = ScanSegmenter(model, 3.0, -25.0)
  knn = KNN()
  tta = TTA(flip=True, shifts=(0, 256, 37))
  res = seg.segment_device(pts, offsets, want_point_labels=True, knn=knn, tta=tta)
  proj = seg.projector.project(pts, offsets, empty_fill=0.0, want_point_outputs=True)
  merged = forward_tta(model, proj["image"], tta)
  assert torch.equal(res["predictions"], merged["predictions"])
  plain = seg.segment_device(pts, offsets, want_point_labels=True, knn=knn)
  assert not torch.equal(res["predictions"], plain["predictions"]), "six views should change some pixels"
  offs = offsets.cpu().numpy()
  win, valid = PL.winner_range(proj["keys"].cpu().numpy(), offs, proj["unproj_range"].cpu().numpy())
  want = PL.point_labels_batch(res["predictions"].cpu().numpy(), win, valid, offs, proj["proj_x"].cpu().numpy(),
                               proj["proj_y"].cpu().numpy(), proj["unproj_range"].cpu().numpy(), mc.NUM_CLASS,
                               mc.CLASSES.index("None"), search=5, k=5, weights=knn.weights(), cutoff=1.0,
                               ignore_class=knn.ignore_index(mc))
  assert np.array_equal(res["point_labels"].cpu().numpy(), want)


def _write_kitti(tmp_path, rng, sizes):
  scan_dir, lab_dir = tmp_path / "velodyne", tmp_path / "labels"
  scan_dir.mkdir()
  lab_dir.mkdir()
  for i, n in enumerate(sizes):
    synth_scan(rng, n).tofile(str(scan_dir / ("%06d.bin" % i)))
    rng.integers(0, 11, n).astype(np.uint32).tofile(str(lab_dir / ("%06d.label" % i)))
  return scan_dir, lab_dir


def test_scan_evaluator_with_tta(tmp_path, small_model):
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  from pclsegmentation_b200.tta import TTA
  mc, model = small_model
  rng = np.random.default_rng(11)
  scan_dir, lab_dir = _write_kitti(tmp_path, rng, [9000, 7000, 5000])
  files = sorted(str(p) for p in scan_dir.iterdir())
  labs = sorted(str(p) for p in lab_dir.iterdir())
  knn, tta = KNN(), TTA(shifts=(0, 128))
  ev = ScanEvaluator(model, 3.0, -25.0, knn=knn, tta=tta)
  loader = ScanBatchLoader("kitti")
  cm = np.zeros((mc.NUM_CLASS, mc.NUM_CLASS), np.int64)
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2], labs[lo:lo + 2])
    res = ev.update(data)
    want = ev.seg.segment_device(data["points"], data["offsets"], want_point_labels=True, knn=knn, tta=tta)
    assert torch.equal(res["point_labels"], want["point_labels"])
    gt = res["gt"].cpu().numpy().astype(np.int64)
    cm += np.bincount(gt * mc.NUM_CLASS + res["point_labels"].cpu().numpy(),
                      minlength=mc.NUM_CLASS ** 2).reshape(mc.NUM_CLASS, mc.NUM_CLASS)
  rep = ev.finish()
  assert np.array_equal(rep["confusion_matrix"], cm) and cm.sum() == 21000


# ---- CLIs ----

@pytest.fixture(scope="module")
def golden(golden_dir):
  with np.load(os.path.join(golden_dir, "nn_sample_dataset.npz")) as f:
    return {k: f[k] for k in f.files}


def _sample_model(tmp_path):
  from pclsegmentation_b200.utils.args_loader import load_model_config
  mc, model = load_model_config("squeezesegv2", "squeezesegv2")
  model.randomize_batch_norm(1)
  wpath = str(tmp_path / "weights.npz")
  model.save_weights_npz(wpath)
  return mc, model, wpath


def test_inference_and_eval_cli_with_tta(tmp_path, golden, capsys):
  from pclsegmentation_b200 import eval as ev
  from pclsegmentation_b200 import inference
  from pclsegmentation_b200.tta import TTA, forward_tta
  mc, model, wpath = _sample_model(tmp_path)
  d = tmp_path / "data" / "val"
  d.mkdir(parents=True)
  for n, f in zip(golden["names"], golden["frames"]):
    np.save(str(d / str(n)), f.astype(np.float64))
  tta = TTA(flip=True, shifts=(0, 120))
  frames = torch.from_numpy(golden["frames"].astype(np.float32)).cuda()
  want = forward_tta(model, frames, tta)["predictions"].cpu().numpy()
  outdir = tmp_path / "out"
  inference.main(["-d", str(d / "*.npy"), "-m", "squeezesegv2", "-n", "squeezesegv2", "-t", str(outdir), "-p", wpath,
                  "-b", "2", "--no_plots", "--tta", "--tta_shifts", "0,120"])
  for i, n in enumerate(golden["names"]):
    pred = np.load(str(outdir / ("pred_" + os.path.splitext(str(n))[0] + ".npy")))
    assert np.array_equal(pred, want[i])
  plain = model.forward_device(frames, None, mean=mc.INPUT_MEAN, std=mc.INPUT_STD)["predictions"].cpu().numpy()
  assert not np.array_equal(plain, want)
  rep = ev.main(["-d", str(tmp_path / "data"), "-i", "val", "-m", "squeezesegv2", "-n", "squeezesegv2", "-p", wpath,
                 "-b", "2", "--tta", "--tta_shifts", "0,120"])
  assert "MIoU:" in capsys.readouterr().out
  cm = C.confusion_matrix(golden["label"].astype(np.int32), want, mc.NUM_CLASS)
  assert np.array_equal(rep["confusion_matrix"], cm)


def test_segment_scans_cli_with_tta(tmp_path, capsys):
  from pclsegmentation_b200 import segment_scans
  from pclsegmentation_b200.dataset_convert import ScanBatchLoader
  from pclsegmentation_b200.pipeline import KNN, ScanEvaluator
  from pclsegmentation_b200.tta import TTA
  from pclsegmentation_b200.utils.args_loader import load_model_config
  rng = np.random.default_rng(12)
  scan_dir, lab_dir = _write_kitti(tmp_path, rng, [8000, 6000, 7000])
  out = tmp_path / "pred"
  args = ["--scans", str(scan_dir / "*.bin"), "-m", "squeezesegv2", "-n", "squeezesegv2kitti", "--random_init",
          "--batch", "2", "--output_dir", str(out), "--tta", "--tta_shifts", "0,512"]
  rep_cli = segment_scans.main(args + ["--labels", str(lab_dir / "*.label")])
  capsys.readouterr()
  mc, model = load_model_config("squeezesegv2", "squeezesegv2kitti")     # the CLI's model: same seeded init
  assert mc.AZIMUTH_LEVEL == 1024
  ev = ScanEvaluator(model, 3.0, -25.0, knn=KNN(), tta=TTA(shifts=(0, 512)))
  loader = ScanBatchLoader("kitti")
  files = sorted(str(p) for p in scan_dir.iterdir())
  labs = sorted(str(p) for p in lab_dir.iterdir())
  for lo in (0, 2):
    data = loader.load(files[lo:lo + 2], labs[lo:lo + 2])
    res = ev.update(data)
    for f, lab in zip(files[lo:lo + 2], ev.seg.point_labels(res, data["sizes"])):
      got = np.fromfile(str(out / (os.path.splitext(os.path.basename(f))[0] + ".label")), dtype=np.uint32)
      assert np.array_equal(got, lab.astype(np.uint32))
  assert np.array_equal(rep_cli["confusion_matrix"], ev.finish()["confusion_matrix"])
