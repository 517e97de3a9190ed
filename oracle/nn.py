"""CPU restatement (PyTorch-CPU, fp32 or fp64) of the reference's network forward
(TEST INFRASTRUCTURE ONLY - never imported by the product).

PARITY UNPINNED: the reference's arithmetic for this part lives in
tensorflow-gpu==2.9.1 (requirements.txt:1; not vendored, not installable here) and the
reference holds no tests / golden logits / weights.  This file restates the published
TF/Keras 2.9 semantics (SURVEY.md Appendix B) for exactly the graph the reference builds:

* ``SqueezeSegV2.call`` + ``CAM/FIRE/FIREUP.call``   pcl_segmentation/nets/SqueezeSegV2.py:285-325, 66-70, 123-127, 191-199
  (layers constructed at :232-283)
* ``Darknet.call`` + ``BasicBlock/EncoderLayer/DecoderLayer.call``  pcl_segmentation/nets/Darknet.py:279-314, 54-66, 96-103, 130-138
  (stride rewriting :158-181, :216-231; ``model_blocks`` :142-145; skip bookkeeping :263-277)
* ``PCLSegmentationNetwork.segmentation_head``      pcl_segmentation/nets/SegmentationNetwork.py:58-69
* input stage ``inference.py:47-72`` == ``DataLoader.parse_sample`` data_loader/data_loader.py:153-187

Weights are a flat dict keyed by Keras attribute paths (SURVEY.md Appendix C), e.g.
``"fire2/squeeze/kernel"`` ``[1,1,64,16]``, ``"enc3/residual_1/bn2/moving_variance"``.
BatchNorm is applied UNFOLDED here (eps = 1e-3, the Keras default - no ``epsilon=`` is passed
anywhere in the reference), so the product's host-side folding is actually tested.
Activations are NHWC at the interface like the reference; NCHW internally.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

BN_EPS = 1e-3  # tf.keras.layers.BatchNormalization default

MODEL_BLOCKS = {21: [1, 1, 2, 2, 1], 53: [1, 2, 8, 8, 4]}  # nets/Darknet.py:142-145


# --------------------------------------------------------------------------------------
# TF 'SAME' primitives
# --------------------------------------------------------------------------------------
def same_pad(n_in: int, k: int, s: int):
    """TF SAME: out = ceil(in/s); total = max((out-1)*s + k - in, 0); before = total//2."""
    n_out = -(-n_in // s)
    total = max((n_out - 1) * s + k - n_in, 0)
    return total // 2, total - total // 2


def conv2d_same(x, kernel, bias=None, strides=(1, 1)):
    """tf.keras.layers.Conv2D(padding='SAME'); x NCHW; kernel Keras layout [kh,kw,Cin,Cout]."""
    kh, kw = kernel.shape[0], kernel.shape[1]
    pt, pb = same_pad(x.shape[2], kh, strides[0])
    pl, pr = same_pad(x.shape[3], kw, strides[1])
    x = F.pad(x, (pl, pr, pt, pb))
    w = kernel.permute(3, 2, 0, 1).contiguous()
    return F.conv2d(x, w, bias, stride=strides)


def conv2d_transpose_1x4_s2(x, kernel, bias=None):
    """tf.keras.layers.Conv2DTranspose(kernel_size=[1,4], strides=[1,2], padding='SAME');
    kernel Keras layout [1,4,Cout,Cin]; out[m] = b + sum_{m = 2j + k - 1} in[j] * w[k]."""
    w = kernel.permute(3, 2, 0, 1).contiguous()  # [Cin, Cout, 1, 4], no spatial flip
    return F.conv_transpose2d(x, w, bias, stride=(1, 2), padding=(0, 1))


def max_pool_same(x, k, strides):
    """tf max-pool, padding='SAME' (padding never wins the max)."""
    pt, pb = same_pad(x.shape[2], k, strides[0])
    pl, pr = same_pad(x.shape[3], k, strides[1])
    x = F.pad(x, (pl, pr, pt, pb), value=float("-inf"))
    return F.max_pool2d(x, kernel_size=k, stride=strides)


def batch_norm(x, p, prefix):
    g = p[prefix + "/gamma"].view(1, -1, 1, 1)
    b = p[prefix + "/beta"].view(1, -1, 1, 1)
    m = p[prefix + "/moving_mean"].view(1, -1, 1, 1)
    v = p[prefix + "/moving_variance"].view(1, -1, 1, 1)
    return g * (x - m) / torch.sqrt(v + BN_EPS) + b


def _conv(x, p, name, strides=(1, 1)):
    return conv2d_same(x, p[name + "/kernel"], p.get(name + "/bias"), strides)


def leaky(x):
    return F.leaky_relu(x, 0.1)


# --------------------------------------------------------------------------------------
# SqueezeSegV2  (nets/SqueezeSegV2.py)
# --------------------------------------------------------------------------------------
def cam(x, p, name):  # CAM.call :66-70
    pool = max_pool_same(x, 7, (1, 1))
    sq = F.relu(batch_norm(_conv(pool, p, name + "/squeeze"), p, name + "/squeeze_bn"))
    ex = torch.sigmoid(batch_norm(_conv(sq, p, name + "/excitation"), p, name + "/excitation_bn"))
    return x * ex


def fire(x, p, name):  # FIRE.call :123-127
    sq = F.relu(batch_norm(_conv(x, p, name + "/squeeze"), p, name + "/squeeze_bn"))
    e1 = F.relu(batch_norm(_conv(sq, p, name + "/expand1x1"), p, name + "/expand1x1_bn"))
    e3 = F.relu(batch_norm(_conv(sq, p, name + "/expand3x3"), p, name + "/expand3x3_bn"))
    return torch.cat([e1, e3], dim=1)


def fireup(x, p, name):  # FIREUP.call :191-199 (stride 2 everywhere in the graph)
    sq = F.relu(batch_norm(_conv(x, p, name + "/squeeze"), p, name + "/squeeze_bn"))
    up = F.relu(conv2d_transpose_1x4_s2(sq, p[name + "/upconv/kernel"], p[name + "/upconv/bias"]))  # no BN
    e1 = F.relu(batch_norm(_conv(up, p, name + "/expand1x1"), p, name + "/expand1x1_bn"))
    e3 = F.relu(batch_norm(_conv(up, p, name + "/expand3x3"), p, name + "/expand3x3_bn"))
    return torch.cat([e1, e3], dim=1)


def squeezesegv2_logits(lidar_nchw, p, taps=None):
    """SqueezeSegV2.call :285-323 up to the logits."""
    t = {} if taps is None else taps
    x = F.relu(batch_norm(_conv(lidar_nchw, p, "conv1", (1, 2)), p, "bn1"))
    cam1 = cam(x, p, "cam1")
    skip = batch_norm(_conv(lidar_nchw, p, "conv1_skip"), p, "bn1_skip")  # no activation (:293)
    t["conv1"], t["cam1"], t["conv1_skip"] = x, cam1, skip
    x = max_pool_same(cam1, 3, (1, 2))
    x = fire(x, p, "fire2")
    t["fire2"] = x
    x = cam(x, p, "cam2")
    x = fire(x, p, "fire3")
    cam3 = cam(x, p, "cam3")
    t["cam3"] = cam3
    x = max_pool_same(cam3, 3, (1, 2))
    x = fire(x, p, "fire4")
    fire5 = fire(x, p, "fire5")
    t["fire5"] = fire5
    x = max_pool_same(fire5, 3, (1, 2))
    x = fire(x, p, "fire6")
    x = fire(x, p, "fire7")
    x = fire(x, p, "fire8")
    fire9 = fire(x, p, "fire9")
    t["fire9"] = fire9
    x = fireup(fire9, p, "fire10") + fire5
    t["fire10"] = x
    x = fireup(x, p, "fire11") + cam3
    x = fireup(x, p, "fire12") + cam1
    x = fireup(x, p, "fire13") + skip
    t["fire13"] = x
    return _conv(x, p, "conv14")  # dropout is identity at inference (:321)


# --------------------------------------------------------------------------------------
# Darknet  (nets/Darknet.py)
# --------------------------------------------------------------------------------------
def darknet_strides(output_stride: int):
    """Restates the stride rewriting at nets/Darknet.py:158-181 (encoder) and :216-231 (decoder)."""
    enc = [2, 2, 2, 2, 2]
    cur = 1
    for s in enc:
        cur *= s
    if output_stride <= cur:
        for i, s in enumerate(reversed(enc)):
            if int(cur) != output_stride:
                if s == 2:
                    cur /= 2
                    enc[-1 - i] = 1
                if int(cur) == output_stride:
                    break
    dec = [2, 2, 2, 2, 2]
    cur = 1
    for s in dec:
        cur *= s
    for i, s in enumerate(dec):
        if int(cur) != output_stride:
            if s == 2:
                cur /= 2
                dec[i] = 1
            if int(cur) == output_stride:
                break
    return enc, dec


def basic_block(x, p, name):  # BasicBlock.call :54-66
    y = leaky(batch_norm(_conv(x, p, name + "/conv1"), p, name + "/bn1"))
    y = leaky(batch_norm(_conv(y, p, name + "/conv2"), p, name + "/bn2"))
    return y + x


def encoder_layer(x, p, name, nblocks, stride):  # EncoderLayer.call :96-103
    x = leaky(batch_norm(_conv(x, p, name + "/conv1", (1, stride)), p, name + "/bn1"))
    for i in range(nblocks):
        x = basic_block(x, p, f"{name}/residual_{i}")
    return x


def decoder_layer(x, p, name, stride):  # DecoderLayer.call :130-138
    if stride == 2:
        x = conv2d_transpose_1x4_s2(x, p[name + "/upconv1/kernel"], p[name + "/upconv1/bias"])
    else:
        x = _conv(x, p, name + "/conv1")
    x = leaky(batch_norm(x, p, name + "/bn1"))
    return basic_block(x, p, name + "/block")


def darknet_logits(lidar_nchw, p, num_layers=53, output_stride=16, taps=None):
    """Darknet.call :279-312 up to the logits, incl. the ``skips``/``os`` bookkeeping of
    run_enc_block / run_dec_block (:263-277)."""
    t = {} if taps is None else taps
    enc_s, dec_s = darknet_strides(output_stride)
    nb = MODEL_BLOCKS[num_layers]
    skips, os_ = {}, 1
    x = leaky(batch_norm(_conv(lidar_nchw, p, "conv1"), p, "bn1"))
    t["conv1"] = x
    for i in range(5):
        y = encoder_layer(x, p, f"enc{i + 1}", nb[i], enc_s[i])
        if y.shape[2] < x.shape[2] or y.shape[3] < x.shape[3]:
            skips[os_] = x
            os_ *= 2
        x = y
        t[f"enc{i + 1}"] = x
    for j, i in enumerate([5, 4, 3, 2, 1]):
        y = decoder_layer(x, p, f"dec{i}", dec_s[j])
        if y.shape[3] > x.shape[3]:
            os_ //= 2
            y = y + skips[os_]
        x = y
        t[f"dec{i}"] = x
    return _conv(x, p, "head")


# --------------------------------------------------------------------------------------
# head / input stage / public entry
# --------------------------------------------------------------------------------------
def segmentation_head(logits_nhwc, mask, none_index):
    """SegmentationNetwork.py:58-69: softmax -> argmax over the *probabilities* (first index on
    ties) -> int32 -> where(mask, pred, CLASSES.index('None')).  Probabilities are not masked."""
    prob = torch.softmax(logits_nhwc, dim=-1)
    pred = torch.argmax(prob, dim=-1).to(torch.int32)
    pred = torch.where(mask.bool(), pred, torch.full_like(pred, int(none_index)))
    return prob, pred


def input_stage(sample_hw6, mean, std, none_index):
    """inference.py:47-72 / data_loader.py:153-187.  sample [H,W,6] (x,y,z,i,d,label) ->
    lidar [H,W,6] float32 (5 normalised channels computed in float64 + mask), mask [H,W] bool,
    label [H,W] int32 (None at empty pixels)."""
    sample = np.asarray(sample_hw6).astype(np.float32)
    lidar = sample[:, :, :5]
    mask = lidar[:, :, 4] > 0
    lidar = (lidar - np.asarray(mean, np.float64).reshape(1, 1, 5)) / np.asarray(std, np.float64).reshape(1, 1, 5)
    lidar[~mask] = 0.0
    lidar = np.append(lidar, np.expand_dims(mask, -1), axis=2)
    return lidar.astype(np.float32), mask, label_to_int32(fixed_label(sample, none_index))


def fixed_label(sample_hw6, none_index):
    """data_loader.py:176-178: the float32 label channel with label[~mask] = none_index.  parse_sample keeps it float
    until its return, so the class-weight map (class_weight_map) compares this float label, not the int32 cast."""
    sample = np.asarray(sample_hw6).astype(np.float32)
    label = sample[..., 5].copy()
    label[~(sample[..., 4] > 0)] = none_index
    return label


def label_to_int32(label):
    """label.astype('int32') (data_loader.py:187) with the rule pclseg.h states for pcls_input_stage: truncation toward
    zero, saturated to the int32 range, NaN -> 0.  numpy's own cast leaves NaN and out-of-range values to the host
    (INT_MIN on x86); on integer-valued labels in range both agree."""
    x = np.asarray(label, dtype=np.float64)
    x = np.where(np.isnan(x), 0.0, np.clip(np.trunc(x), -2.0 ** 31, 2.0 ** 31 - 1))
    return x.astype(np.int32)


def to_torch_params(params: dict, dtype=torch.float32):
    return {k: torch.as_tensor(np.asarray(v)).to(dtype) for k, v in params.items()}


@torch.no_grad()
def forward(arch: str, params: dict, lidar_bhw6, mask_bhw, none_index: int,
            num_layers: int = 53, output_stride: int = 16, dtype=torch.float32, taps=None):
    """model([lidar, mask]) -> (logits, probabilities, predictions), all NHWC numpy.

    arch: 'squeezesegv2' | 'darknet'.  lidar is the already-normalised 6-channel input
    (inference.py:56-62), mask bool [B,H,W]."""
    p = {k: (v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v))).to(dtype) for k, v in params.items()}
    x = torch.as_tensor(np.asarray(lidar_bhw6)).to(dtype).permute(0, 3, 1, 2).contiguous()
    if arch == "squeezesegv2":
        logits = squeezesegv2_logits(x, p, taps)
    elif arch == "darknet":
        logits = darknet_logits(x, p, num_layers, output_stride, taps)
    else:
        raise ValueError(arch)
    logits = logits.permute(0, 2, 3, 1).contiguous()
    prob, pred = segmentation_head(logits, torch.as_tensor(np.asarray(mask_bhw)), none_index)
    return logits.numpy(), prob.numpy(), pred.numpy()


def class_weight_map(label_hw, cls_loss_weight):
    """data_loader.py:181-185: weight = zeros(label.shape); weight[label == l] = CLS_LOSS_WEIGHT[l] for l in
    range(NUM_CLASS); returned as float32 like parse_sample (:187).  label_hw is the FLOAT label of fixed_label, as
    parse_sample compares it: 2.5, NaN and +-inf match no class (weight 0), -0.0 matches class 0."""
    weight = np.zeros(np.asarray(label_hw).shape)
    for l in range(len(cls_loss_weight)):
        weight[np.asarray(label_hw) == l] = cls_loss_weight[int(l)]
    return weight.astype("float32")
