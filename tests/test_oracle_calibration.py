"""Calibrated confidence without a GPU: known answers of the float64 oracle (oracle/calibration.py), the temperature
fit on planted temperatures, the argument checks of the four C entry points, ``Calibration`` / TTA refusals and the
two-rank gloo reduce of the accumulators."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import calibration as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.calibration import Calibration, check_tta, fit_temperature, inv_temperature
from pclsegmentation_b200.metrics import reliability_scores


def test_uniform_logits_give_conf_one_over_nc_and_entropy_one():
  for nc in (2, 11, 20, 32):
    z = np.full((5, nc), 3.25, np.float32)
    p, conf, ent = O.confidence(logits=z, a=np.float32(0.7))
    assert np.allclose(p, 1.0 / nc, rtol=0, atol=1e-15)
    assert np.allclose(conf, 1.0 / nc, rtol=0, atol=1e-15) and np.allclose(ent, 1.0, rtol=0, atol=1e-12)
  _, conf, ent = O.confidence(logits=np.zeros((3, 1), np.float32))
  assert (conf == 1.0).all() and (ent == 0.0).all()
  _, conf, ent = O.confidence(logits=np.random.default_rng(0).normal(0, 3, (4, 20)).astype(np.float32),
                              mask=np.array([1, 0, 1, 0]))
  assert conf[1] == conf[3] == ent[1] == ent[3] == 0.0 and conf[0] > 0


def test_confidence_does_not_increase_with_temperature():
  z = np.random.default_rng(1).normal(0, 4, (2000, 20)).astype(np.float32)
  prev = None
  for T in (0.25, 0.5, 1.0, 1.5, 2.0, 3.7, 8.0):
    _, conf, _ = O.confidence(logits=z, a=O.inv_temperature(T))
    if prev is not None:
      assert (conf <= prev + 1e-15).all(), T
    prev = conf


def test_ece_of_a_calibrated_and_of_an_always_wrong_construction():
  # per bin: confidence c exactly and a fraction c of the elements correct
  nb = 10
  conf, pred, label = [], [], []
  for k, c in enumerate([0.05, 0.25, 0.5, 0.75, 1.0]):
    n = 40
    ncor = int(round(c * n))
    conf += [c] * n
    pred += [1] * n
    label += [1] * ncor + [2] * (n - ncor)
  cnt, cor, cs = O.reliability(np.array(conf, np.float32), pred, label, 5, -1, nb)
  ece, mce = O.ece_mce(cnt, cor, cs)
  assert cnt.sum() == 200 and ece < 1e-7 and mce < 1e-7
  rep = reliability_scores(cnt, cor, cs)
  assert rep["ece"] < 1e-7 and rep["count"] == 200 and rep["accuracy"] == pytest.approx(cor.sum() / 200)
  # every prediction wrong at confidence 1: ECE = MCE = 1
  cnt, cor, cs = O.reliability(np.ones(50, np.float32), np.zeros(50), np.ones(50), 3, -1, 15)
  assert O.ece_mce(cnt, cor, cs) == (1.0, 1.0) and cnt[-1] == 50
  rep = reliability_scores(cnt, cor, cs)
  assert rep["ece"] == rep["mce"] == 1.0 and rep["accuracy"] == 0.0 and rep["mean_confidence"] == 1.0


def test_bin_rule_and_counting():
  nb = 15
  edges = (np.arange(nb + 1) / nb).astype(np.float32)
  b = O.bin_index(edges, nb)
  want = np.minimum(np.trunc(edges * np.float32(nb)), nb - 1).astype(np.int64)
  assert np.array_equal(b, want) and b[-1] == nb - 1 and b[0] == 0
  assert O.bin_index(np.array([-0.5, 0.0, 1.0, 1.5], np.float32), 4).tolist() == [0, 0, 3, 3]
  # labels / predictions outside [0, NC) and the ignored class are not counted
  cnt, cor, cs = O.reliability(np.full(6, 0.5, np.float32), [0, 1, -1, 2, 1, 5], [0, 1, 1, 4, -3, 2], 5, 4, 2)
  assert cnt.tolist() == [0, 2] and cor.tolist() == [0, 2] and cs[1] == 1.0


def test_parabola_vertex_of_an_exact_quadratic():
  t = O.log_grid(0.25, 4.0, 64)
  x0 = np.log(1.37)
  nll = 2.5 * (np.log(t) - x0) ** 2 + 0.8
  t_star, edge = fit_temperature(t, nll)
  assert not edge and t_star == pytest.approx(1.37, rel=1e-12)
  assert O.fit(t, nll)[0] == pytest.approx(1.37, rel=1e-9)
  assert Calibration().grid_temperatures()[0] == 0.25 and Calibration().grid_temperatures()[-1] == 4.0
  assert np.allclose(Calibration().grid_temperatures(), t, rtol=1e-15, atol=0)


def test_edge_flag_at_both_grid_ends():
  t = O.log_grid(0.25, 4.0, 16)
  assert fit_temperature(t, np.log(t)) == (0.25, True)
  assert fit_temperature(t, -np.log(t)) == (4.0, True)
  assert O.fit(t, np.log(t)) == (0.25, True) and O.fit(t, -np.log(t)) == (4.0, True)
  assert fit_temperature(t, (np.log(t) - np.log(t[1])) ** 2)[1] is False


@pytest.mark.parametrize("T0", [0.5, 1.0, 2.0])
def test_planted_temperature_is_recovered(T0):
  """Labels drawn from softmax(z / T0): the NLL grid's fit lands within 2 % of T0."""
  rng = np.random.default_rng(int(T0 * 100))
  n, nc = 200_000, 20
  z = rng.normal(0, 3, (n, nc)).astype(np.float32)
  p = O.softmax(z, O.inv_temperature(T0))
  label = (rng.random(n)[:, None] > np.cumsum(p, 1)).sum(1).clip(0, nc - 1)
  cal = Calibration(fit=True)
  temps = cal.grid_temperatures()
  sums, count, _ = O.temperature_nll(z, label, nc, -1, [inv_temperature(T) for T in temps])
  assert count == n
  t_star, edge = fit_temperature(temps, sums / count)
  assert not edge and abs(t_star / T0 - 1) < 0.02, t_star


def test_nll_counts_only_class_labels_and_matches_a_direct_softmax():
  rng = np.random.default_rng(3)
  z = rng.normal(0, 2, (300, 11)).astype(np.float32)
  label = rng.integers(-2, 13, 300)
  label[::7] = 4
  sums, count, bound = O.temperature_nll(z, label, 11, 4, [np.float32(0.5), np.float32(1.0)])
  ok = (label >= 0) & (label < 11) & (label != 4)
  assert count == ok.sum()
  p = O.softmax(z[ok], np.float32(0.5))
  assert sums[0] == pytest.approx(-np.log(p[np.arange(ok.sum()), label[ok]]).sum(), rel=1e-12)
  assert (bound > 0).all()


def test_point_confidence_oracle():
  probs = np.random.default_rng(4).random((2, 3, 4, 5)).astype(np.float32)
  offsets = np.array([0, 3, 5])
  px = np.array([0, -1, 3, 2, 1])
  py = np.array([2, 0, 1, 0, 2])
  lab = np.array([4, 1, 5, 0, -1])
  got = O.point_confidence(probs, offsets, px, py, lab)
  assert got.tolist() == [probs[0, 2, 0, 4], 0.0, 0.0, probs[1, 0, 2, 0], 0.0]


def test_calibration_arguments():
  Calibration(temperature=0.3, n_bins=64, grid=(0.1, 10.0, 2))
  for kw, msg in ((dict(temperature=0.0), "temperature"), (dict(temperature=-1.0), "temperature"),
                  (dict(temperature=float("inf")), "temperature"), (dict(temperature=float("nan")), "temperature"),
                  (dict(n_bins=0), "n_bins"), (dict(n_bins=65), "n_bins"), (dict(grid=(0.25, 4.0, 1)), "points"),
                  (dict(grid=(0.25, 4.0, 65)), "points"), (dict(grid=(4.0, 0.25, 8)), "lo < hi"),
                  (dict(grid=(0.0, 4.0, 8)), "lo < hi")):
    with pytest.raises(ValueError, match=msg):
      Calibration(**kw)
  assert inv_temperature(3.0) == float(np.float32(1.0 / 3.0))


def test_tta_with_a_temperature_or_a_fit_is_refused():
  from pclsegmentation_b200.tta import TTA
  check_tta(Calibration(), TTA())
  check_tta(Calibration(temperature=2.0), None)
  for cal in (Calibration(temperature=2.0), Calibration(fit=True)):
    with pytest.raises(ValueError, match="merges probabilities"):
      check_tta(cal, TTA())


# ---- C argument checks ----

def _f32(v):
  return (ctypes.c_float * len(v))(*v)


def test_argument_validation_without_gpu():
  lib = _lib.load()

  def conf(logits=1, probs=None, nc=20, a=1.0, out=(None, 1, None)):
    return lib.pcls_confidence(logits, probs, None, 10, nc, a, *out, None)

  for kw, msg in ((dict(nc=33), b"num_classes"), (dict(nc=0), b"num_classes"), (dict(probs=1), b"exactly one"),
                  (dict(logits=None), b"exactly one"), (dict(logits=None, probs=1, a=0.5), b"probs mode"),
                  (dict(a=0.0), b"inv_temperature"), (dict(a=-1.0), b"inv_temperature"),
                  (dict(a=float("inf")), b"inv_temperature"), (dict(a=float("nan")), b"inv_temperature"),
                  (dict(out=(None, None, None)), b"no output")):
    assert conf(**kw) == -1, kw
    assert b"pcls_confidence" in lib.pcls_last_error() and msg in lib.pcls_last_error(), (kw, lib.pcls_last_error())

  def nll(nc=20, temps=(1.0, 0.5), n_temps=None, label=1):
    t = _f32(list(temps)) if temps is not None else None
    return lib.pcls_temperature_nll(1, label, 10, nc, -1, len(temps or ()) if n_temps is None else n_temps, t, 1, 1, None)

  for kw, msg in ((dict(nc=33), b"num_classes"), (dict(temps=(), n_temps=0), b"n_temps"),
                  (dict(temps=(1.0,) * 65), b"n_temps"), (dict(temps=None, n_temps=3), b"NULL"),
                  (dict(temps=(1.0, 0.0)), b"inverse temperature 1"), (dict(temps=(float("nan"),)), b"inverse temperature 0"),
                  (dict(label=None), b"NULL")):
    assert nll(**kw) == -1, kw
    assert b"pcls_temperature_nll" in lib.pcls_last_error() and msg in lib.pcls_last_error(), (kw, lib.pcls_last_error())

  def rel(nc=20, bins=15, cnt=1):
    return lib.pcls_reliability_update(1, 1, 1, 10, nc, -1, bins, cnt, 1, 1, None)

  for kw, msg in ((dict(nc=33), b"num_classes"), (dict(bins=0), b"n_bins"), (dict(bins=65), b"n_bins"),
                  (dict(cnt=None), b"NULL")):
    assert rel(**kw) == -1, kw
    assert b"pcls_reliability_update" in lib.pcls_last_error() and msg in lib.pcls_last_error(), kw

  def pc(B=1, nc=20, out=1, total=10):
    return lib.pcls_point_confidence(1, 1, B, 4, 8, total, 1, 1, 1, nc, out, None)

  for kw, msg in ((dict(nc=33), b"num_classes"), (dict(B=-1), b"bad sizes"), (dict(B=0), b"no scan"),
                  (dict(out=None), b"NULL")):
    assert pc(**kw) == -1, kw
    assert b"pcls_point_confidence" in lib.pcls_last_error() and msg in lib.pcls_last_error(), kw
  # n == 0 is a no-op once the arguments are valid (no device needed)
  assert lib.pcls_confidence(1, None, None, 0, 20, 0.5, None, 1, None, None) == 0
  assert lib.pcls_temperature_nll(None, None, 0, 20, -1, 2, _f32([1.0, 2.0]), None, None, None) == 0
  assert lib.pcls_reliability_update(None, None, None, 0, 20, -1, 15, None, None, None, None) == 0
  assert lib.pcls_point_confidence(None, None, 0, 4, 8, 0, None, None, None, 20, None, None) == 0


# ---- two-rank gloo reduce of the accumulators ----

def _free_port():
  with socket.socket() as s:
    s.bind(("127.0.0.1", 0))
    return s.getsockname()[1]


def _worker(rank, world, port, parts, out):
  os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
  dist.init_process_group("gloo", rank=rank, world_size=world)
  try:
    from pclsegmentation_b200.metrics import Reliability
    from pclsegmentation_b200.sharding import Communicator
    cnt, cor, cs, nll, n = parts[rank]
    rel = Reliability(15, 20)
    rel.count, rel.correct, rel.conf = torch.from_numpy(cnt), torch.from_numpy(cor), torch.from_numpy(cs)
    nll_t, n_t = torch.from_numpy(nll), torch.tensor([n], dtype=torch.int64)
    comm = Communicator()
    rel.allreduce(comm)
    comm.allreduce_sums([nll_t, n_t])
    out[rank] = (rel.result(), nll_t.numpy().copy(), int(n_t.item()))
  finally:
    dist.destroy_process_group()


def test_two_rank_reduce_of_the_accumulators():
  rng = np.random.default_rng(5)
  conf = rng.random(4000).astype(np.float32)
  pred, label = rng.integers(0, 20, 4000), rng.integers(-1, 21, 4000)
  z = rng.normal(0, 2, (4000, 20)).astype(np.float32)
  temps = [inv_temperature(T) for T in Calibration().grid_temperatures()]
  parts = []
  for lo, hi in ((0, 2100), (2100, 4000)):
    cnt, cor, cs = O.reliability(conf[lo:hi], pred[lo:hi], label[lo:hi], 20, 19, 15)
    sums, n, _ = O.temperature_nll(z[lo:hi], label[lo:hi], 20, 19, temps)
    parts.append((cnt, cor, cs, sums, n))
  mgr = mp.Manager()
  out = mgr.dict()
  mp.spawn(_worker, args=(2, _free_port(), parts, out), nprocs=2, join=True)
  cnt, cor, cs = O.reliability(conf, pred, label, 20, 19, 15)
  sums, n, _ = O.temperature_nll(z, label, 20, 19, temps)
  want = reliability_scores(cnt, cor, cs)
  for r in range(2):
    rep, nll, count = out[r]
    assert np.array_equal(rep["bin_count"], cnt) and np.array_equal(rep["bin_accuracy"], want["bin_accuracy"])
    assert np.allclose(rep["bin_confidence"], want["bin_confidence"], rtol=1e-12, atol=0)
    assert rep["ece"] == pytest.approx(want["ece"], rel=1e-12) and count == n
    assert np.allclose(nll, sums, rtol=1e-12, atol=0)
