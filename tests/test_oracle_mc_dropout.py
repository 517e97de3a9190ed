"""MC dropout without a GPU: the Philox generator against Random123's known answers, the statistics of the masks, the
thr / scale rules, the accumulate / finalize rules, the binned AUROC, ``MCDropout`` validation, the C argument checks
and the dropout sites the model builders record."""
import math

import numpy as np
import pytest

from oracle import mc_dropout as O
from pclsegmentation_b200 import _lib
from pclsegmentation_b200.metrics import binned_auroc
from pclsegmentation_b200.mc_dropout import MCDropout, check_exclusive, dropout_threshold


@pytest.mark.parametrize("ctr,key,want", [
  ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
  ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
  ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
   [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])])
def test_philox_known_answers(ctr, key, want):
  assert [int(v) for v in O.philox4x32_10(np.array(ctr), np.array(key))] == want


@pytest.mark.parametrize("rate", [0.01, 0.1, 0.5])
def test_keep_rate_within_4_sigma(rate):
  n = 10_000_000
  u = O.uniforms(seed=12345, frame=7, n_pass=3, site=1, n_elements=n)
  p = 1.0 - O.threshold(rate) / 65536.0
  kept = float((u >= O.threshold(rate)).mean())
  assert abs(kept - p) <= 4 * math.sqrt(p * (1 - p) / n), (kept, p)


@pytest.mark.parametrize("other", [dict(frame=8), dict(n_pass=4), dict(site=2), dict(seed=12346),
                                   dict(frame=7 + (1 << 32))])
def test_masks_of_different_keys_are_independent(other):
  rate, n = 0.3, 2_000_000
  base = dict(seed=12345, frame=7, n_pass=3, site=1)
  thr = O.threshold(rate)
  a = O.uniforms(n_elements=n, **base) >= thr
  b = O.uniforms(n_elements=n, **{**base, **other}) >= thr
  r = thr / 65536.0
  q = r * r + (1 - r) * (1 - r)
  agree = float((a == b).mean())
  assert abs(agree - q) <= 4 * math.sqrt(q * (1 - q) / n), (agree, q)


def test_element_order_within_a_philox_call():
  """Output word i's low half goes to element 8g + 2i, its high half to element 8g + 2i + 1."""
  w = O.philox4x32_10(np.array([[1, 5 | (2 << 16), 9, 0]]), np.array([3, 0]))[0]
  u = O.uniforms(seed=3, frame=9, n_pass=2, site=5, n_elements=16)
  want = [int(w[i]) >> (16 * j) & 0xFFFF for i in range(4) for j in range(2)]
  assert list(u[8:16]) == want


def test_rate_zero_is_the_identity_and_threshold_edges():
  rng = np.random.default_rng(0)
  bits = rng.integers(0, 1 << 16, (2, 3, 4, 8), dtype=np.uint16)
  for dt in ("f16", "bf16"):
    finite = np.isfinite(O.to_f32(bits, dt))
    got = O.dropout_bits(bits, dt, 1, 0, 0, 0, 0.0)
    assert np.array_equal(got[finite], bits[finite])
  assert O.threshold(0.0) == 0 and O.scale_of(0) == np.float32(1.0)
  assert O.threshold(0.5) == 32768 and O.scale_of(32768) == np.float32(2.0)
  assert O.threshold(1.5 / 65536) == 2                          # ties round up: floor(x + 0.5)
  assert O.threshold(65535.4 / 65536) == 65535
  with pytest.raises(ValueError):
    O.threshold(65535.5 / 65536)                                # thr = 65536 would drop everything
  assert dropout_threshold(0.1) == O.threshold(0.1) == 6554
  assert O.scale_of(6554) == np.float32(65536.0 / (65536 - 6554))


def test_dropout_bits_keep_rule_and_values():
  rng = np.random.default_rng(1)
  x = rng.normal(0, 3, (2, 2, 5, 16)).astype(np.float32)
  for dt in ("f16", "bf16"):
    bits = O.from_f32(x, dt)
    got = O.dropout_bits(bits, dt, 99, 4, 1, 2, 0.25)
    keep = O.keep_mask(99, 4, 1, 2, 0.25, bits.shape)
    assert (got[~keep] == 0).all()
    scaled = O.to_f32(bits, dt) * np.float32(65536 / (65536 - 16384))
    assert np.array_equal(got[keep], O.from_f32(scaled, dt)[keep])
    assert 0.6 < keep.mean() < 0.9


def test_bf16_rounding_is_round_to_nearest_even():
  vals = np.array([1.0, 1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, -2.5, 1e-40], np.float32)
  got = O.to_f32(O.from_f32(vals, "bf16"), "bf16")
  assert list(got[:4]) == [1.0, 1.0, 1.0 + 2 ** -6, -2.5]


def test_accumulate_finalize_known_answers():
  nc = 4
  p0 = np.array([[0.25, 0.25, 0.25, 0.25], [0.7, 0.1, 0.1, 0.1], [0.5, 0.5, 0.0, 0.0]], np.float32)
  p1 = np.array([[0.25, 0.25, 0.25, 0.25], [0.1, 0.7, 0.1, 0.1], [0.5, 0.5, 0.0, 0.0]], np.float32)
  # T = 1: the mean is the probabilities unchanged, MI = 0
  a, h = O.accumulate([p0])
  r = O.finalize(a, h, None, 1, 3)
  assert np.array_equal(r["probabilities"], p0) and (r["mutual_information"] == 0).all()
  assert list(r["predictions"]) == [0, 0, 0]                   # planted ties: the first index
  # T = 2: disagreement gives MI > 0 on pixel 1 only
  a, h = O.accumulate([p0, p1])
  r = O.finalize(a, h, np.array([1, 1, 0], np.uint8), 2, 3)
  assert list(r["predictions"]) == [0, 0, 3]                   # pixel 1 ties 0.4 / 0.4; pixel 2 is masked
  assert r["mutual_information"][0] == 0 and r["mutual_information"][1] > 0.1 and r["mutual_information"][2] == 0
  assert r["confidence"][2] == 0 and r["entropy"][2] == 0
  assert abs(r["entropy"][0] - 1.0) < 1e-6
  # equal passes (rate 0): T = 2 gives the pass's bits back and MI = 0 exactly; from T = 3 on the running float32 sum
  # rounds (3p is not exact), so T = 8 is only close
  a, h = O.accumulate([p1] * 2)
  r = O.finalize(a, h, None, 2, 3)
  assert np.array_equal(r["probabilities"], p1) and (r["mutual_information"] == 0).all()
  a, h = O.accumulate([p1] * 8)
  r = O.finalize(a, h, None, 8, 3)
  assert np.abs(r["probabilities"] - p1).max() <= 8 * np.finfo(np.float32).eps
  assert not np.array_equal(r["probabilities"], p1)
  a, h = O.accumulate([p0, p1, p0])
  assert np.array_equal(a, ((p0 + p1).astype(np.float32) + p0).astype(np.float32))
  r = O.finalize(a, h, None, 3, 3)
  assert np.array_equal(r["probabilities"], (a / np.float32(3)).astype(np.float32))
  assert nc == a.shape[-1]


def test_binned_auroc_known_answers():
  # perfect separation: every error in a higher bin than every correct element
  assert binned_auroc([5, 0, 3], [5, 0, 0]) == 1.0
  assert O.binned_auroc([5, 0, 3], [5, 0, 0]) == 1.0
  assert binned_auroc([3, 0, 5], [0, 0, 5]) == 0.0          # reversed
  assert binned_auroc([0, 10, 0], [0, 4, 0]) == 0.5         # all in one bin
  assert binned_auroc([4, 4], [4, 4]) == 0.5                # no errors
  c, k = np.array([7, 3, 5, 9]), np.array([6, 2, 1, 0])
  assert binned_auroc(c, k) == pytest.approx(O.binned_auroc(c, k))
  # brute force over pairs
  err_bins = np.repeat(np.arange(4), c - k)
  ok_bins = np.repeat(np.arange(4), k)
  pairs = (err_bins[:, None] > ok_bins[None, :]) + 0.5 * (err_bins[:, None] == ok_bins[None, :])
  assert binned_auroc(c, k) == pytest.approx(pairs.mean())


def test_mcdropout_validation():
  m = MCDropout(passes=4, seed=(1 << 64) - 1, rate=0.5)
  assert m.next_frame == 0 and m.passes == 4
  for kw in (dict(passes=0), dict(passes=257), dict(seed=-1), dict(seed=1 << 64), dict(rate=-0.1),
             dict(rate=1.0), dict(rate=float("nan"))):
    with pytest.raises(ValueError):
      MCDropout(**kw)

  class Cfg:
    DROP_RATE = 0.1
  assert MCDropout().rate_for(Cfg) == 0.1
  assert MCDropout(rate=0.0).rate_for(Cfg) == 0.0

  class Cal:
    temperature, fit = 1.0, False
  check_exclusive(MCDropout(), None, Cal)
  Cal.temperature = 2.0
  with pytest.raises(ValueError):
    check_exclusive(MCDropout(), None, Cal)
  with pytest.raises(ValueError):
    check_exclusive(MCDropout(), object(), None)


def test_c_argument_checks_without_gpu():
  lib = _lib.load()

  def acc(nc=20, pss=0, p=1, out=1):
    return lib.pcls_mc_accumulate(p, 10, nc, pss, out, 1, None)

  for kw, msg in ((dict(nc=33), b"num_classes"), (dict(nc=0), b"num_classes"), (dict(pss=-1), b"pass"),
                  (dict(pss=65536), b"pass"), (dict(p=None), b"NULL"), (dict(out=None), b"NULL")):
    assert acc(**kw) == -1, kw
    assert b"pcls_mc_accumulate" in lib.pcls_last_error() and msg in lib.pcls_last_error(), kw

  def fin(nc=20, none=0, T=4, acc_p=1, outs=(None, 1, None, None, None)):
    return lib.pcls_mc_finalize(acc_p, 1, None, 10, nc, none, T, *outs, None)

  for kw, msg in ((dict(nc=33), b"num_classes"), (dict(none=20), b"none_index"), (dict(T=0), b"n_passes"),
                  (dict(T=65537), b"n_passes"), (dict(outs=(None,) * 5), b"no output"), (dict(acc_p=None), b"NULL")):
    assert fin(**kw) == -1, kw
    assert b"pcls_mc_finalize" in lib.pcls_last_error() and msg in lib.pcls_last_error(), kw
  assert lib.pcls_mc_accumulate(None, 0, 20, 0, None, None, None) == 0
  assert lib.pcls_mc_finalize(None, None, None, 0, 20, 0, 1, None, 1, None, None, None, None) == 0
  assert lib.pcls_net_dropout(None, 1, 0, 0.1) == -1 and b"pcls_net_dropout" in lib.pcls_last_error()
  assert lib.pcls_net_set_dropout(None, 0, 0, 0, None) == -1 and b"pcls_net_set_dropout" in lib.pcls_last_error()


@pytest.mark.parametrize("name,cfg,n_sites,channels", [("squeezesegv2", "squeezesegv2kitti", 1, [64]),
                                                       ("darknet21", "darknet21", 6, None),
                                                       ("darknet53", "darknet53kitti", 6, None)])
def test_dropout_sites_and_unchanged_program(name, cfg, n_sites, channels):
  from pclsegmentation_b200.utils.args_loader import config_map, model_map
  mc = config_map[cfg]()
  mc.ZENITH_LEVEL, mc.AZIMUTH_LEVEL = 32, 256
  model = model_map[name](mc)
  g = model._graph
  assert len(g.dropout_sites) == n_sites
  assert all(rate == mc.DROP_RATE for _, rate, _ in g.dropout_sites)
  if channels is not None:
    assert [s.channels for s, _, _ in g.dropout_sites] == channels
    assert g.dropout_sites[0][0] is model._taps["fire13"] and g.dropout_sites[0][0].width == 256
  else:
    assert [s for s, _, _ in g.dropout_sites[:5]] == [model._taps["enc%d" % i] for i in range(1, 6)]
    assert g.dropout_sites[5][0] is model._taps["dec1"]
  assert all(s.channels % 8 == 0 for s, _, _ in g.dropout_sites)
  # the program holds no dropout op: the default net's pcls_net_* call sequence is what it was
  assert all(op["op"] in ("conv", "pool", "cam") for op in g.program)
  positions = [next(i for i, op in enumerate(g.program) if op is after) for _, _, after in g.dropout_sites]
  assert positions == sorted(positions) and positions[-1] == len(g.program) - 2   # the last site feeds the logits conv
  assert all(after["dst"] is sym for sym, _, after in g.dropout_sites)          # each follows its tensor's producer


def test_site_behind_a_replaced_op_is_refused():
  """A site whose op left the program (e.g. merged away after the Dropout call) is an error at build time, not a
  dropout emitted at a shifted position."""
  from pclsegmentation_b200.nets.layers import Graph
  g = Graph(4, 16)
  x = g.conv(g.input, "c1", _lib.KIND_CONV, 1, 1, 1, 16, True)
  g.dropout(x, 0.1)
  y = g.conv(x, "c2", _lib.KIND_CONV, 1, 1, 1, 8, True)
  g.program[0] = dict(g.program[0])                        # the op the site follows is replaced
  with pytest.raises(ValueError, match="no longer in the program"):
    g.build_net(y, 8, 0, 0, 1, dropout_rate=0.1)
