// pcls_net: op-list executor for the SqueezeSegV2 / Darknet forward (sm_100a).
//
// The Python model builders describe the graph (pcls_net_tensor / _conv / _maxpool3x3_s2 / _cam); this file
// folds BatchNorm into the convolutions, packs weights, plans the activation arena by liveness and runs the ops
// on a stream (optionally as a replayed CUDA graph).  Replaces model([lidar, mask]) == SqueezeSegV2.call
// (pcl_segmentation/nets/SqueezeSegV2.py:285-325) / Darknet.call (nets/Darknet.py:279-314) + segmentation_head
// (nets/SegmentationNetwork.py:58-69).
#include "net.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace pcls {

int pad48_mode = 1;   // A/B switch (pcls_net_set_option "pad48", before the ops are added)
int pair_s2_mode = 1; // A/B switch "pair_s2": stride-2 convs with Cin = 32 run on the pixel-pair view (build_pair_view)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

template <typename T>
static void pack_to(std::vector<uint16_t>& dst, const std::vector<float>& src) {
  dst.resize(src.size());
  for (size_t i = 0; i < src.size(); ++i) {
    if (sizeof(T) == 2 && std::is_same<T, __half>::value) {
      __half h = __float2half_rn(src[i]);
      memcpy(&dst[i], &h, 2);
    } else {
      __nv_bfloat16 h = __float2bfloat16_rn(src[i]);
      memcpy(&dst[i], &h, 2);
    }
  }
}

// y = gamma * (conv + b - mean) / sqrt(var + eps) + beta  ==  conv * scale + bias'
static void fold_bn(int cout, const float* b, const float* gamma, const float* beta, const float* mean,
                    const float* var, float eps, std::vector<double>& scale, std::vector<double>& bias) {
  scale.assign(cout, 1.0);
  bias.assign(cout, 0.0);
  for (int c = 0; c < cout; ++c) {
    const double b0 = b ? (double)b[c] : 0.0;
    if (gamma) {
      const double sc = (double)gamma[c] / std::sqrt((double)var[c] + (double)eps);
      scale[c] = sc;
      bias[c] = (b0 - (double)mean[c]) * sc + (double)beta[c];
    } else {
      bias[c] = b0;
    }
  }
}

int Net::add_tensor(int width, int channels, bool logits) {
  TensorInfo t;
  t.width = width;
  t.channels = channels;
  t.stride = channels;
  t.logits = logits;
  tensors.push_back(t);
  return (int)tensors.size() - 1;
}

size_t Net::tensor_frame_bytes(const TensorInfo& t) const {
  return (size_t)H * t.width * t.stride * (t.logits ? 4 : 2);
}

int Net::add_conv(const pcls_conv_desc& d) {
  PCLS_REQUIRE(!finalized, "pcls_net_conv: net already finalized");
  ConvLayer L;
  if (d.kind == PCLS_CONV) {
    if (d.kh == 1 && d.kw == 1 && d.stride_w == 1) L.p.mode = MODE_1x1;
    else if (d.kh == 3 && d.kw == 3 && d.stride_w == 1) L.p.mode = MODE_3x3_S1;
    else if (d.kh == 3 && d.kw == 3 && d.stride_w == 2) L.p.mode = MODE_3x3_S2;
    else PCLS_REQUIRE(false, "pcls_net_conv: unsupported Conv2D %dx%d stride_w %d", d.kh, d.kw, d.stride_w);
  } else if (d.kind == PCLS_DECONV_1x4_S2) {
    PCLS_REQUIRE(d.kh == 1 && d.kw == 4 && d.stride_w == 2, "pcls_net_conv: transposed conv must be [1,4] stride [1,2]");
    L.p.mode = MODE_DECONV;
  } else {
    PCLS_REQUIRE(false, "pcls_net_conv: unknown kind %d", d.kind);
  }
  PCLS_REQUIRE(d.in_tensor >= 0 && d.in_tensor < (int)tensors.size() && d.out_tensor > 0 &&
                   d.out_tensor < (int)tensors.size() && d.in_tensor != d.out_tensor,
               "pcls_net_conv: bad tensor ids in=%d out=%d", d.in_tensor, d.out_tensor);
  // Channel padding 48 -> 64 (fire6 / fire7 squeeze outputs): with 48 channels the tcgen05 path has to walk K in
  // 16-channel chunks (32-byte TMA / UMMA rows: nine 4 KB loads per tile, measured 0.21 of the HBM roofline for the 3x3
  // expand); stored with a 64-channel pixel stride the tensor takes the 128-byte-row path like every other layer.  The
  // producing conv writes all 64 channels (zero weights and bias beyond 48: act(0) = 0), consumers contract 64 input
  // channels against zero-padded kernels.  Only for tensors that ONE convolution writes completely.
  if (pad48_mode && !tensors[d.out_tensor].logits && tensors[d.out_tensor].channels == 48 && tensors[d.out_tensor].stride == 48 &&
      d.out_channel_offset == 0 && d.cout == 48 && d.residual0 < 0 && d.residual1 < 0 && d.kind == PCLS_CONV)
    tensors[d.out_tensor].stride = 64;
  const TensorInfo& ti = tensors[d.in_tensor];
  const TensorInfo& to = tensors[d.out_tensor];
  PCLS_REQUIRE(!ti.logits, "pcls_net_conv: cannot read a logits tensor");
  PCLS_REQUIRE(d.cin >= 1 && d.cin <= ti.channels && d.cout >= 1, "pcls_net_conv: cin %d exceeds input tensor channels %d",
               d.cin, ti.channels);
  PCLS_REQUIRE(d.out_channel_offset >= 0 && d.out_channel_offset + d.cout <= to.channels,
               "pcls_net_conv: output slice [%d,%d) exceeds tensor channels %d", d.out_channel_offset,
               d.out_channel_offset + d.cout, to.channels);
  PCLS_REQUIRE((d.out_is_logits != 0) == to.logits, "pcls_net_conv: out_is_logits does not match the output tensor");
  PCLS_REQUIRE(to.logits || d.out_channel_offset % 8 == 0, "pcls_net_conv: channel offset must be a multiple of 8");
  int wout = ti.width;
  if (L.p.mode == MODE_3x3_S2) wout = (ti.width + 1) / 2;
  if (L.p.mode == MODE_DECONV) wout = ti.width * 2;
  PCLS_REQUIRE(to.width == wout, "pcls_net_conv: output width %d, expected %d", to.width, wout);
  PCLS_REQUIRE(d.h_kernel != nullptr, "pcls_net_conv: kernel is NULL");
  const bool bn = d.h_bn_gamma != nullptr;
  PCLS_REQUIRE(!bn || (d.h_bn_beta && d.h_bn_mean && d.h_bn_var), "pcls_net_conv: incomplete BatchNorm parameters");
  PCLS_REQUIRE(d.act >= 0 && d.act <= 2, "pcls_net_conv: bad activation %d", d.act);
  const int res[2] = {d.residual0, d.residual1};
  for (int r = 0; r < 2; ++r) {
    if (res[r] < 0) continue;
    PCLS_REQUIRE(res[r] < (int)tensors.size() && !tensors[res[r]].logits && tensors[res[r]].width == to.width &&
                     d.out_channel_offset + d.cout <= tensors[res[r]].channels && res[r] != d.out_tensor,
                 "pcls_net_conv: residual tensor %d does not match the output", res[r]);
  }

  ConvParams& p = L.p;
  p.H = H; p.Win = ti.width; p.Wout = wout;
  const bool in_padded = ti.stride > ti.channels, out_padded = to.stride > to.channels;
  p.cin = d.cin; p.cin_pad = in_padded ? ti.stride : (d.cin + 15) / 16 * 16;
  p.in_channels = ti.stride;
  p.cout = out_padded ? to.stride : d.cout; p.cout_pad = (p.cout + 15) / 16 * 16;
  p.out_channels = to.stride; p.out_coff = d.out_channel_offset;
  L.cin_logical = d.cin; L.cout_logical = d.cout;
  p.act = d.act;
  p.ntaps = (p.mode == MODE_1x1) ? 1 : (p.mode == MODE_DECONV ? 4 : 9);
  p.pad_left = 0;
  if (p.mode == MODE_3x3_S2) {
    const int total = std::max((wout - 1) * 2 + 3 - ti.width, 0);
    p.pad_left = total / 2;
  }
  p.out_f32 = d.out_is_logits ? 1 : 0;
  p.res0_channels = d.residual0 >= 0 ? tensors[d.residual0].stride : 0;
  p.res1_channels = d.residual1 >= 0 ? tensors[d.residual1].stride : 0;
  L.in = d.in_tensor; L.out = d.out_tensor; L.res0 = d.residual0; L.res1 = d.residual1;

  // fold BN, pack [tap][cout_pad][cin_pad]
  std::vector<double> scale, bias;
  fold_bn(d.cout, d.h_bias, d.h_bn_gamma, d.h_bn_beta, d.h_bn_mean, d.h_bn_var, d.bn_eps, scale, bias);
  L.w_f32.assign((size_t)p.ntaps * p.cout_pad * p.cin_pad, 0.0f);
  for (int t = 0; t < p.ntaps; ++t)
    for (int co = 0; co < d.cout; ++co)
      for (int ci = 0; ci < d.cin; ++ci) {
        const size_t src = (d.kind == PCLS_CONV) ? ((size_t)t * d.cin + ci) * d.cout + co   // [kh,kw,Cin,Cout]
                                                 : ((size_t)t * d.cout + co) * d.cin + ci;  // [1,4,Cout,Cin]
        L.w_f32[((size_t)t * p.cout_pad + co) * p.cin_pad + ci] = (float)((double)d.h_kernel[src] * scale[co]);
      }
  L.bias_f32.assign(p.cout_pad, 0.0f);
  for (int co = 0; co < d.cout; ++co) L.bias_f32[co] = (float)bias[co];

  build_pair_view(L);
  convs.push_back(std::move(L));
  ops.push_back({OP_CONV, (int)convs.size() - 1});
  return PCLS_OK;
}

// The 8-channel network input viewed as pixel pairs [B,H,W/2,16] turns the three kinds of input convolution into
// shapes the tcgen05 kernel runs (K chunk 16):
//   1x1 (SqueezeSegV2 conv1_skip)        -> 1x1 on pairs, block-diagonal weights, N = 2 Cout (both pixels of the pair)
//   3x3 s1 (Darknet conv1)               -> 3x3 on pairs, N = 2 Cout; pixel 2j+p, tap kx reads pair j+dw, parity par
//                                           with kx = 2 dw + par - p + 1
//   3x3 s[1,2], even W (SqueezeSegV2 conv1) -> 6 taps (dh, dw in {0,1}); kx = 0,1 live in pair wo, kx = 2 in pair wo+1
// Weights that fall outside the 3x3 support are zero; outputs are bit-identical in layout ([..,W,C] == [..,W/2,2C]).
// Transposed [1,4] / stride [1,2] convolution as ONE 3-tap GEMM producing both output parities:
//   out[2j]   = in[j] w1 + in[j-1] w3        out[2j+1] = in[j+1] w0 + in[j] w2
// => N = 2 Cout, taps dw = -1: [w3 | 0], dw = 0: [w1 | w2], dw = +1: [0 | w0]; the output tensor [.., 2W, C]
// (channel offset 0, C == tensor channels) is the same memory as [.., W, 2C], so stores are contiguous.
void Net::build_deconv_row3(ConvLayer& L) {
  const ConvParams& p = L.p;
  if (p.mode != MODE_DECONV || p.out_f32 || p.out_coff != 0 || p.cout != p.out_channels) return;
  if (2 * p.cout_pad > 256 || p.cout % 8 != 0) return;
  ConvParams q = p;
  q.mode = MODE_ROW3; q.ntaps = 3; q.Wout = p.Win;
  q.cout = 2 * p.cout; q.cout_pad = (q.cout + 15) / 16 * 16; q.out_channels = 2 * p.out_channels;
  q.res0_channels = 2 * p.res0_channels; q.res1_channels = 2 * p.res1_channels;
  auto wf = [&](int tap, int co, int ci) { return L.w_f32[((size_t)tap * p.cout_pad + co) * p.cin_pad + ci]; };
  L.w_tc.assign((size_t)3 * q.cout_pad * p.cin_pad, 0.0f);
  auto put = [&](int t, int half, int k) {
    for (int co = 0; co < p.cout; ++co)
      for (int ci = 0; ci < p.cin; ++ci)
        L.w_tc[((size_t)t * q.cout_pad + half * p.cout + co) * p.cin_pad + ci] = wf(k, co, ci);
  };
  put(0, 0, 3); put(1, 0, 1); put(1, 1, 2); put(2, 1, 0);
  L.bias_tc.assign(q.cout_pad, 0.0f);
  for (int n = 0; n < q.cout; ++n) L.bias_tc[n] = L.bias_f32[n % p.cout];
  L.ptc = q;
  L.pair_view = true;
}

void Net::build_pair_view(ConvLayer& L) {
  const ConvParams& p = L.p;
  if (p.mode == MODE_DECONV) { build_deconv_row3(L); return; }
  // 3x3 s[1,2] deeper in the net (Darknet's enc1.down 32 -> 64 and enc2.down 64 -> 128): as a strided convolution every tap
  // is its own TMA box of 128 rows x Cin channels taken from every other pixel (64-byte rows for Cin = 32) - nine loads per
  // tile, and the wait-cycle counters show the MMA issuer waiting for data 54 % of the kernel at 0.24 of the HBM peak.  On
  // the pixel-pair view [B,H,W/2,2 Cin] the layer is a 3x3 stride-1 convolution whose dw = -1 taps are zero: three
  // 130-pair halo tiles with 128-byte rows per tile: enc1.down 0.328 -> 0.202 ms at batch 32.  A third of the MMAs multiply
  // zeros and the zero taps' weights are loaded like any others: for Cin = 64 (enc2.down, 295 KB of pair-view weights
  // streamed per tile) the same change measured 0.219 -> 0.343 ms, so Cin = 32 only.
  if (L.in != 0 && pair_s2_mode && p.mode == MODE_3x3_S2 && p.pad_left == 0 && p.Win % 2 == 0 && !p.out_f32 && L.res0 < 0 &&
      L.res1 < 0 && p.cin == p.cin_pad && p.in_channels == p.cin_pad && p.cin_pad == 32 && p.Wout == p.Win / 2) {
    ConvParams q = p;
    const int cp2 = 2 * p.cin_pad;
    q.Win = p.Win / 2; q.in_channels = cp2; q.cin = cp2; q.cin_pad = cp2; q.pad_left = 0;
    q.mode = MODE_3x3_S1; q.ntaps = 9;
    L.w_tc.assign((size_t)9 * q.cout_pad * cp2, 0.0f);
    for (int dh = 0; dh < 3; ++dh)
      for (int kx = 0; kx < 3; ++kx)
        for (int co = 0; co < p.cout; ++co)
          for (int ci = 0; ci < p.cin; ++ci)
            L.w_tc[((size_t)(dh * 3 + 1 + (kx >> 1)) * q.cout_pad + co) * cp2 + (kx & 1) * p.cin_pad + ci] =
                L.w_f32[((size_t)(dh * 3 + kx) * p.cout_pad + co) * p.cin_pad + ci];
    L.bias_tc = L.bias_f32;
    L.ptc = q;
    L.pair_view = true;
    return;
  }
  if (L.in != 0 || W % 2 != 0 || p.out_f32 || L.res0 >= 0 || L.res1 >= 0) return;
  if (p.mode == MODE_3x3_S2 && p.pad_left != 0) return;
  if (p.mode == MODE_DECONV) return;
  const bool doubled = p.mode != MODE_3x3_S2;
  if (doubled && (p.out_coff != 0 || p.cout != p.out_channels)) return;
  ConvParams q = p;
  q.Win = W / 2; q.Wout = W / 2; q.in_channels = 16; q.cin = 16; q.cin_pad = 16; q.pad_left = 0;
  const int co_n = p.cout;
  if (doubled) { q.cout = 2 * co_n; q.out_channels = 2 * p.out_channels; }
  q.cout_pad = (q.cout + 15) / 16 * 16;
  if (q.cout_pad > 256) return;
  auto wf = [&](int tap, int co, int ci) { return L.w_f32[((size_t)tap * p.cout_pad + co) * p.cin_pad + ci]; };
  if (p.mode == MODE_1x1) {
    q.mode = MODE_1x1; q.ntaps = 1;
    L.w_tc.assign((size_t)q.cout_pad * 16, 0.0f);
    for (int px = 0; px < 2; ++px)
      for (int co = 0; co < co_n; ++co)
        for (int ci = 0; ci < p.cin; ++ci) L.w_tc[(size_t)(px * co_n + co) * 16 + px * 8 + ci] = wf(0, co, ci);
  } else if (p.mode == MODE_3x3_S1) {
    q.mode = MODE_3x3_S1; q.ntaps = 9;
    L.w_tc.assign((size_t)9 * q.cout_pad * 16, 0.0f);
    for (int dh = 0; dh < 3; ++dh)
      for (int dw = -1; dw <= 1; ++dw)
        for (int px = 0; px < 2; ++px)
          for (int par = 0; par < 2; ++par) {
            const int kx = 2 * dw + par - px + 1;
            if (kx < 0 || kx > 2) continue;
            for (int co = 0; co < co_n; ++co)
              for (int ci = 0; ci < p.cin; ++ci)
                L.w_tc[((size_t)(dh * 3 + dw + 1) * q.cout_pad + px * co_n + co) * 16 + par * 8 + ci] = wf(dh * 3 + kx, co, ci);
          }
  } else {
    // 3x3 s[1,2] on pairs: kx = 0,1 live in pair wo (dw = 0), kx = 2 in pair wo + 1 (dw = +1).  Expressed as a 3x3
    // stride-1 convolution on the pair tensor whose dw = -1 taps are zero, so that it takes the halo / pixel-group
    // path of the tensor-core kernel (128-byte TMA rows) instead of six 32-byte-row loads per tile.
    q.mode = MODE_3x3_S1; q.ntaps = 9;
    L.w_tc.assign((size_t)9 * q.cout_pad * 16, 0.0f);
    for (int dh = 0; dh < 3; ++dh)
      for (int kx = 0; kx < 3; ++kx)
        for (int co = 0; co < co_n; ++co)
          for (int ci = 0; ci < p.cin; ++ci)
            L.w_tc[((size_t)(dh * 3 + 1 + (kx >> 1)) * q.cout_pad + co) * 16 + (kx & 1) * 8 + ci] = wf(dh * 3 + kx, co, ci);
  }
  L.bias_tc.assign(q.cout_pad, 0.0f);
  for (int n = 0; n < q.cout; ++n) L.bias_tc[n] = L.bias_f32[n % co_n];
  L.ptc = q;
  L.pair_view = true;
}

int Net::add_pool(int in, int out) {
  PCLS_REQUIRE(!finalized, "pcls_net_maxpool3x3_s2: net already finalized");
  PCLS_REQUIRE(in >= 0 && in < (int)tensors.size() && out > 0 && out < (int)tensors.size() && in != out,
               "pcls_net_maxpool3x3_s2: bad tensor ids");
  const TensorInfo &ti = tensors[in], &to = tensors[out];
  PCLS_REQUIRE(!ti.logits && !to.logits && ti.channels == to.channels && to.width == (ti.width + 1) / 2,
               "pcls_net_maxpool3x3_s2: shape mismatch");
  tensors[out].stride = tensors[in].stride;   // a padded input (zero pads) pools into a padded output
  PoolLayer L;
  L.in = in; L.out = out;
  L.pad_left = std::max((to.width - 1) * 2 + 3 - ti.width, 0) / 2;
  pools.push_back(L);
  ops.push_back({OP_POOL, (int)pools.size() - 1});
  return PCLS_OK;
}

int Net::add_cam(const pcls_cam_desc& d) {
  PCLS_REQUIRE(!finalized, "pcls_net_cam: net already finalized");
  PCLS_REQUIRE(d.in_tensor >= 0 && d.in_tensor < (int)tensors.size() && d.out_tensor > 0 &&
                   d.out_tensor < (int)tensors.size() && d.in_tensor != d.out_tensor,
               "pcls_net_cam: bad tensor ids");
  const TensorInfo &ti = tensors[d.in_tensor], &to = tensors[d.out_tensor];
  PCLS_REQUIRE(ti.channels == d.channels && to.channels == d.channels && ti.width == to.width && !ti.logits && !to.logits,
               "pcls_net_cam: shape mismatch");
  PCLS_REQUIRE((d.channels == 64 || d.channels == 128) && d.reduced == d.channels / 16,
               "pcls_net_cam: supported channels 64/128 with reduction 16 (got %d -> %d)", d.channels, d.reduced);
  PCLS_REQUIRE(d.h_sq_kernel && d.h_ex_kernel, "pcls_net_cam: kernels must not be NULL");
  CamLayer L;
  L.in = d.in_tensor; L.out = d.out_tensor; L.C = d.channels; L.R = d.reduced;
  std::vector<double> s1, bb1, s2, bb2;
  fold_bn(L.R, d.h_sq_bias, d.h_sq_gamma, d.h_sq_beta, d.h_sq_mean, d.h_sq_var, d.bn_eps, s1, bb1);
  fold_bn(L.C, d.h_ex_bias, d.h_ex_gamma, d.h_ex_beta, d.h_ex_mean, d.h_ex_var, d.bn_eps, s2, bb2);
  L.h.resize((size_t)2 * L.C * L.R + L.R + L.C);
  float* w1 = L.h.data();           // [C][R]  Keras [1,1,C,R]
  float* w2 = w1 + L.C * L.R;       // [R][C]  Keras [1,1,R,C]
  float* b1 = w2 + L.R * L.C;
  float* b2 = b1 + L.R;
  for (int c = 0; c < L.C; ++c)
    for (int j = 0; j < L.R; ++j) w1[c * L.R + j] = (float)((double)d.h_sq_kernel[c * L.R + j] * s1[j]);
  for (int j = 0; j < L.R; ++j)
    for (int c = 0; c < L.C; ++c) w2[j * L.C + c] = (float)((double)d.h_ex_kernel[j * L.C + c] * s2[c]);
  for (int j = 0; j < L.R; ++j) b1[j] = (float)bb1[j];
  for (int c = 0; c < L.C; ++c) b2[c] = (float)bb2[c];
  cams.push_back(std::move(L));
  ops.push_back({OP_CAM, (int)cams.size() - 1});
  return PCLS_OK;
}

void Net::op_tensors(const OpRef& op, std::vector<int>& reads, std::vector<int>& writes) const {
  reads.clear(); writes.clear();
  if (op.type == OP_CONV) {
    const ConvLayer& L = convs[op.index];
    if (L.skip_into >= 0) return;   // computed by the conv that reads its output: neither reads nor writes
    reads.push_back(L.in);
    if (L.pool_src >= 0) reads.push_back(L.pool_src);   // (fused max-pool: the un-pooled tensor is what the kernel reads)
    if (L.up_squeeze >= 0) reads.push_back(convs[L.up_squeeze].in);   // (fused squeeze conv: its input is what the kernel reads)
    if (L.skip_src >= 0) reads.push_back(convs[L.skip_src].in);      // (fused skip: computed from the network input)
    else if (L.res0 >= 0) reads.push_back(L.res0);
    if (L.res1 >= 0) reads.push_back(L.res1);
    writes.push_back(L.out);
  } else if (op.type == OP_POOL) {
    reads.push_back(pools[op.index].in); writes.push_back(pools[op.index].out);
  } else {
    reads.push_back(cams[op.index].in); writes.push_back(cams[op.index].out);
  }
}

int Net::finalize(int logits_tensor_, int num_classes_, int none_index_) {
  PCLS_REQUIRE(!finalized, "pcls_net_finalize: already finalized");
  PCLS_REQUIRE(logits_tensor_ > 0 && logits_tensor_ < (int)tensors.size() && tensors[logits_tensor_].logits,
               "pcls_net_finalize: logits tensor id %d is not a logits tensor", logits_tensor_);
  PCLS_REQUIRE(num_classes_ >= 1 && num_classes_ <= 32 && tensors[logits_tensor_].channels == num_classes_ &&
                   tensors[logits_tensor_].width == W,
               "pcls_net_finalize: logits tensor must be [B,H,W,num_classes] with num_classes <= 32");
  PCLS_REQUIRE(none_index_ >= 0 && none_index_ < num_classes_, "pcls_net_finalize: none_index out of range");
  logits_tensor = logits_tensor_; num_classes = num_classes_; none_index = none_index_;

  // max-pool + 1x1 conv fusion (pool_conv.cu): a pool whose output has ONE reader, the 1x1 convolution right behind it
  const int n_ops = (int)ops.size();
  if (fuse_pool)
    for (int i = 0; i + 1 < n_ops; ++i) {
      if (ops[i].type != OP_POOL || ops[i + 1].type != OP_CONV) continue;
      PoolLayer& P = pools[ops[i].index];
      ConvLayer& L = convs[ops[i + 1].index];
      const ConvParams& cp = L.p;
      if (L.in != P.out || cp.mode != MODE_1x1 || L.res0 >= 0 || L.res1 >= 0 || cp.out_f32 || cp.out_coff != 0) continue;
      if (tensors[P.in].stride != tensors[P.in].channels || cp.cin_pad != tensors[P.in].channels) continue;
      if (!pool_conv1x1_supported(tensors[P.in].channels, (L.cout_logical + 15) / 16 * 16) || cp.cout != cp.cout_pad) continue;
      bool other_reader = false;
      std::vector<int> rd, wr;
      for (int k = 0; k < n_ops; ++k) {
        if (k == i + 1) continue;
        op_tensors(ops[k], rd, wr);
        for (int r : rd) other_reader = other_reader || r == P.out;
      }
      if (other_reader) continue;
      P.fused_conv = ops[i + 1].index;
      L.pool_src = P.in; L.pool_pad_left = P.pad_left;
    }
  // squeeze 1x1 + transposed conv fusion (squeeze_upconv.cu): the squeeze output has ONE reader, the [1,4]/s[1,2] transposed
  // conv right behind it (FIREUP).  Not with keep_tensors: the squeeze tensor is then never written.
  if (fuse_up && !keep_tensors)
    for (int i = 0; i + 1 < n_ops; ++i) {
      if (ops[i].type != OP_CONV || ops[i + 1].type != OP_CONV) continue;
      ConvLayer& Q = convs[ops[i].index];
      ConvLayer& U = convs[ops[i + 1].index];
      const ConvParams &q = Q.p, &u = U.p;
      if (q.mode != MODE_1x1 || u.mode != MODE_DECONV || U.in != Q.out || Q.pool_src >= 0) continue;
      if (Q.res0 >= 0 || Q.res1 >= 0 || U.res0 >= 0 || U.res1 >= 0 || q.out_f32 || u.out_f32 || q.out_coff != 0 || u.out_coff != 0) continue;
      const int C = q.cin_pad, S = q.cout;
      if (tensors[Q.in].stride != C || tensors[Q.in].channels != C || Q.cin_logical != C) continue;
      if (q.cout != q.cout_pad || q.out_channels != S || Q.cout_logical != S) continue;
      if (u.cin_pad != S || u.cout != S || u.cout_pad != S || u.out_channels != S || U.cin_logical != S) continue;
      if (!squeeze_upconv_supported(C, S)) continue;
      bool other_reader = false;
      std::vector<int> rd, wr;
      for (int k = 0; k < n_ops; ++k) {
        if (k == i + 1) continue;
        op_tensors(ops[k], rd, wr);
        for (int r : rd) other_reader = other_reader || r == Q.out;
      }
      if (other_reader || Q.out == logits_tensor) continue;
      U.up_squeeze = ops[i].index;
      Q.fused_into_up = ops[i + 1].index;
    }
  // skip fusion (conv_tc.cu, RM = 3): a 1x1 conv of the network input with no activation (SqueezeSegV2's conv1_skip) whose
  // output has ONE reader, a conv that adds it as its residual after the ReLU (fire13's expand), is computed in that
  // conv's epilogue from the 16 bytes per pixel of the input instead of crossing HBM twice at 128 bytes per pixel.  Not
  // with keep_tensors (the skip tensor is then never written) nor with the CUDA-core path.
  if (fuse_skip && !keep_tensors && conv_impl == 0)
    for (int i = 0; i < n_ops; ++i) {
      if (ops[i].type != OP_CONV) continue;
      ConvLayer& P = convs[ops[i].index];
      if (P.in != 0 || P.out == logits_tensor || P.fused_into_up >= 0) continue;
      int reader = -1, n_use = 0;
      std::vector<int> rd, wr;
      for (int k = 0; k < n_ops; ++k) {
        if (k == i) continue;
        op_tensors(ops[k], rd, wr);
        for (int r : rd) if (r == P.out) { ++n_use; reader = k; }
        for (int w : wr) if (w == P.out) n_use += 2;   // a second writer (channel slices) rules it out
      }
      if (n_use != 1 || ops[reader].type != OP_CONV) continue;
      ConvLayer& E = convs[ops[reader].index];
      if (E.pool_src >= 0 || E.up_squeeze >= 0 || !tc_skip_fusable(P, E)) continue;
      E.skip_src = ops[i].index;
      P.skip_into = ops[reader].index;
    }
  // liveness: first write .. last read (op order); the logits tensor lives to the end (head reads it)
  std::vector<int> reads, writes;
  for (auto& t : tensors) { t.first = -1; t.last = -1; }
  tensors[0].first = -1; tensors[0].last = -1;  // input: written by the input kernel before op 0
  for (int i = 0; i < n_ops; ++i) {
    op_tensors(ops[i], reads, writes);
    for (int r : reads) {
      PCLS_REQUIRE(r == 0 || tensors[r].first >= 0, "pcls_net_finalize: op %d reads tensor %d before it is written", i, r);
      tensors[r].last = std::max(tensors[r].last, i);
    }
    for (int w : writes) {
      if (tensors[w].first < 0) tensors[w].first = i;
      tensors[w].last = std::max(tensors[w].last, i);
    }
  }
  tensors[logits_tensor].last = n_ops;
  if (keep_tensors)
    for (auto& t : tensors) t.last = n_ops;

  // greedy first-fit arena planning (per-frame offsets; scaled by the frames per pass)
  struct Block { size_t off, size; };
  std::vector<Block> free_list;
  size_t top = 0;
  auto alloc = [&](size_t size) -> size_t {
    size = align_up(size, 1024);
    for (size_t i = 0; i < free_list.size(); ++i) {
      if (free_list[i].size >= size) {
        size_t off = free_list[i].off;
        free_list[i].off += size; free_list[i].size -= size;
        if (free_list[i].size == 0) free_list.erase(free_list.begin() + i);
        return off;
      }
    }
    size_t off = top; top += size; return off;
  };
  auto release = [&](size_t off, size_t size) {
    size = align_up(size, 1024);
    free_list.push_back({off, size});
    std::sort(free_list.begin(), free_list.end(), [](const Block& a, const Block& b) { return a.off < b.off; });
    for (size_t i = 0; i + 1 < free_list.size();) {
      if (free_list[i].off + free_list[i].size == free_list[i + 1].off) {
        free_list[i].size += free_list[i + 1].size; free_list.erase(free_list.begin() + i + 1);
      } else ++i;
    }
    if (!free_list.empty() && free_list.back().off + free_list.back().size == top) { top = free_list.back().off; free_list.pop_back(); }
  };
  tensors[0].offset = alloc(tensor_frame_bytes(tensors[0]));
  mask_offset = alloc((size_t)H * W);  // u8 mask lives for the whole pass
  size_t peak = top;
  for (int i = 0; i < n_ops; ++i) {
    op_tensors(ops[i], reads, writes);
    for (int w : writes)
      if (tensors[w].first == i) { tensors[w].offset = alloc(tensor_frame_bytes(tensors[w])); peak = std::max(peak, top); }
    // release after the op: tensors whose last use is this op (never the input's slot before its last read)
    for (size_t t = 0; t < tensors.size(); ++t)
      if (tensors[t].last == i && (int)t != logits_tensor && !(t == 0 && tensors[0].last < 0))
        release(tensors[t].offset, tensor_frame_bytes(tensors[t]));
  }
  frame_bytes = align_up(peak, 1024);
  for (size_t t = 0; t < tensors.size(); ++t) {
    bool fused_skip = false;   // (the output of a conv computed by its reader is never materialised)
    for (const auto& L : convs) fused_skip = fused_skip || (L.skip_into >= 0 && L.out == (int)t);
    PCLS_REQUIRE(t == 0 || tensors[t].first >= 0 || fused_skip, "pcls_net_finalize: tensor %d is never written", (int)t);
  }

  frames_per_pass = (micro_batch > 0 && micro_batch < max_batch) ? micro_batch : max_batch;
  PCLS_CHECK_CUDA(cudaMalloc(&arena, frame_bytes * (size_t)frames_per_pass));
  arena_bytes = frame_bytes * (size_t)frames_per_pass;

  // upload weights
  size_t wbytes = 0;
  for (auto& L : convs) {
    wbytes += align_up(L.w_f32.size() * 2, 256) + align_up(L.bias_f32.size() * 4, 256);
    if (L.pair_view) wbytes += align_up(L.w_tc.size() * 2, 256) + align_up(L.bias_tc.size() * 4, 256);
  }
  for (auto& L : cams) wbytes += align_up(L.h.size() * 4, 256);
  PCLS_CHECK_CUDA(cudaMalloc(&weights, std::max<size_t>(wbytes, 256)));
  weight_bytes = wbytes;
  size_t off = 0;
  std::vector<uint16_t> packed;
  for (auto& L : convs) {
    if (precision == PCLS_F16) pack_to<__half>(packed, L.w_f32); else pack_to<__nv_bfloat16>(packed, L.w_f32);
    PCLS_CHECK_CUDA(cudaMemcpy((char*)weights + off, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice));
    L.p.w = (char*)weights + off; off += align_up(packed.size() * 2, 256);
    PCLS_CHECK_CUDA(cudaMemcpy((char*)weights + off, L.bias_f32.data(), L.bias_f32.size() * 4, cudaMemcpyHostToDevice));
    L.p.bias = (const float*)((char*)weights + off); off += align_up(L.bias_f32.size() * 4, 256);
    if (L.pair_view) {
      if (precision == PCLS_F16) pack_to<__half>(packed, L.w_tc); else pack_to<__nv_bfloat16>(packed, L.w_tc);
      PCLS_CHECK_CUDA(cudaMemcpy((char*)weights + off, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice));
      L.ptc.w = (char*)weights + off; off += align_up(packed.size() * 2, 256);
      PCLS_CHECK_CUDA(cudaMemcpy((char*)weights + off, L.bias_tc.data(), L.bias_tc.size() * 4, cudaMemcpyHostToDevice));
      L.ptc.bias = (const float*)((char*)weights + off); off += align_up(L.bias_tc.size() * 4, 256);
    }
  }
  for (auto& L : cams) {
    PCLS_CHECK_CUDA(cudaMemcpy((char*)weights + off, L.h.data(), L.h.size() * 4, cudaMemcpyHostToDevice));
    const float* base = (const float*)((char*)weights + off);
    L.p.C = L.C; L.p.R = L.R;
    L.p.w1 = base; L.p.w2 = base + L.C * L.R; L.p.b1 = L.p.w2 + L.R * L.C; L.p.b2 = L.p.b1 + L.R;
    off += align_up(L.h.size() * 4, 256);
  }
  int rc = tc_prepare();
  if (rc != PCLS_OK) return rc;
  finalized = true;
  return PCLS_OK;
}

void* Net::tensor_ptr(int t, int frames) const {
  // per-pass layout: every tensor is contiguous over the frames of the pass
  (void)frames;
  return (char*)arena + tensors[t].offset * (size_t)frames_per_pass;
}

template <typename T>
int Net::run_pass(const float* lidar, int channels, const uint8_t* mask, bool raw, const double* mean5,
                  const double* std5, int nb, float* logits, float* probs, int32_t* preds, cudaStream_t s,
                  cudaEvent_t* ev) {
  const int64_t n_pixels = (int64_t)nb * H * W;
  pdl_early_now = (pdl_mode && n_pixels <= pdl_early_px) ? 1 : 0;   // small passes: latency mode (common.cuh)
  uint8_t* mask_buf = (uint8_t*)arena + mask_offset * (size_t)frames_per_pass;
  int evi = 0;
  if (ev) cudaEventRecord(ev[evi++], s);
  int rc = PCLS_OK;
  if (lidar != nullptr) {  // (NULL: tensor 0 and the mask were written in place, e.g. by pcls_project_resolve_net_input)
    if (channels & kIn16) rc = launch_net_input16(lidar, channels & ~kIn16, mask, n_pixels, tensor_ptr(0, nb), mask_buf, s);
    else rc = launch_net_input<T>(lidar, channels, mask, raw, mean5, std5, n_pixels, (T*)tensor_ptr(0, nb), mask_buf, s);
  }
  if (rc) return rc;
  float* logits_buf = logits ? logits : (float*)tensor_ptr(logits_tensor, nb);
  bool head_done = false;
  for (const OpRef& op : ops) {
    if (ev) cudaEventRecord(ev[evi++], s);
    if (op.type == OP_CONV) {
      ConvLayer& L = convs[op.index];
      ConvParams p = L.p;
      p.in = tensor_ptr(L.in, nb);
      p.out = (L.out == logits_tensor) ? (void*)logits_buf : tensor_ptr(L.out, nb);
      p.res0 = (L.res0 >= 0 && L.skip_src < 0) ? tensor_ptr(L.res0, nb) : nullptr;   // (fused skip: see TcParams::skip)
      p.res1 = L.res1 >= 0 ? tensor_ptr(L.res1, nb) : nullptr;
      if (conv_impl == 0 && L.fused_into_up >= 0) continue;   // computed by the transposed conv behind it
      if (L.skip_into >= 0) continue;                          // computed in the epilogue of the conv that reads it
      if (conv_impl == 0 && L.up_squeeze >= 0) {
        const ConvLayer& Q = convs[L.up_squeeze];
        SqueezeUpconvParams su;
        su.in = tensor_ptr(Q.in, nb); su.out = p.out;
        su.w1 = Q.p.w; su.b1 = Q.p.bias; su.w1_stride = Q.p.cin_pad; su.act1 = Q.p.act;
        su.w2 = p.w; su.b2 = p.bias; su.w2_cout_pad = p.cout_pad; su.w2_cin_pad = p.cin_pad; su.act2 = p.act;
        su.H = H; su.W = p.Win; su.rows = 0; su.tiles_per_row = 0;
        rc = launch_squeeze_upconv<T>(su, Q.p.cin_pad, Q.p.cout, nb, s);
      } else if (conv_impl == 0 && L.pool_src >= 0) {
        PoolConvParams pc;
        pc.in = tensor_ptr(L.pool_src, nb); pc.out = p.out; pc.w = p.w; pc.bias = p.bias;
        pc.H = H; pc.Win = tensors[L.pool_src].width; pc.Wout = p.Wout; pc.out_channels = p.out_channels;
        pc.w_stride = p.cin_pad; pc.pad_left = L.pool_pad_left; pc.act = p.act; pc.n_strips = 0; pc.tiles_per_row = 0;
        // (a 48 -> 64 padded output: contract the real 48 channels, write the pads as zeros)
        const int S_real = (L.cout_logical + 15) / 16 * 16;
        pc.zero_to = S_real < p.cout ? p.cout : 0;
        rc = launch_pool_conv1x1<T>(pc, tensors[L.pool_src].channels, S_real, nb, s);
      } else if (conv_impl == 0 && L.tc_ok) {
        // the final conv can run the segmentation head in its epilogue (every 32-pixel warp row must be contiguous
        // in memory: full-width tiles of 128 pixels)
        const bool fuse = L.out == logits_tensor && head_is_fused();
        head_args.head = fuse ? 1 : 0;
        head_args.none_index = none_index; head_args.mask = mask_buf;
        head_args.probs = probs; head_args.preds = preds; head_args.logits = logits;
        head_done = head_done || fuse;
        if (L.pair_view) {  // same buffers, re-viewed geometry
          ConvParams pv = L.ptc;
          pv.in = p.in; pv.out = p.out; pv.res0 = p.res0; pv.res1 = p.res1;
          rc = tc_launch(L, pv, nb, s);
        } else {
          rc = tc_launch(L, p, nb, s);
        }
      }
      else rc = launch_conv_direct<T>(p, nb, s);
    } else if (op.type == OP_POOL) {
      const PoolLayer& L = pools[op.index];
      if (conv_impl == 0 && L.fused_conv >= 0) continue;   // pooled on the fly by the 1x1 conv behind it
      rc = launch_maxpool3x3_s2<T>((const T*)tensor_ptr(L.in, nb), (T*)tensor_ptr(L.out, nb), nb, H, tensors[L.in].width,
                                   tensors[L.out].width, tensors[L.in].stride, L.pad_left, s);
    } else {
      const CamLayer& L = cams[op.index];
      rc = launch_cam<T>((const T*)tensor_ptr(L.in, nb), (T*)tensor_ptr(L.out, nb), L.p, nb, H, tensors[L.in].width, cam_px, s);
    }
    if (rc) return rc;
    if (tc_debug_buf && ev && op.type == OP_CONV) {  // development aid: print the counters of this launch
      cudaStreamSynchronize(s);
      std::vector<unsigned long long> h(148 * 24);
      cudaMemcpy(h.data(), tc_debug_buf, h.size() * 8, cudaMemcpyDeviceToHost);
      cudaMemset(tc_debug_buf, 0, h.size() * 8);
      double a[24] = {0};
      for (int c = 0; c < 148; ++c) for (int i = 0; i < 24; ++i) a[i] += (double)h[c * 24 + i] / 148.0;
      const ConvParams& cp = convs[op.index].p;
      fprintf(stderr, "[tc_debug] conv mode %d %dx%d w%d | cycles/CTA: total %.0f | producer wait-empty %.0f | issuer wait-tempty %.0f wait-full %.0f | "
              "epi(g0) wait-tfull %.0f store-drain %.0f barrier %.0f busy %.0f tiles %.0f | epi(g1) wait-tfull %.0f busy %.0f tiles %.0f\n",
              cp.mode, cp.cin, cp.cout, cp.Wout, a[8], a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], a[11], a[14], a[15]);
    }
  }
  if (ev) cudaEventRecord(ev[evi++], s);
  rc = head_done ? PCLS_OK : launch_head(logits_buf, mask_buf, n_pixels, num_classes, none_index, probs, preds, s);
  if (ev) cudaEventRecord(ev[evi++], s);
  return rc;
}

int Net::run_all(const float* lidar, int channels, const uint8_t* mask, bool raw, const double* mean5,
                 const double* std5, int B, float* logits, float* probs, int32_t* preds, cudaStream_t s,
                 cudaEvent_t* ev) {
  const size_t px = (size_t)H * W;
  for (int b0 = 0; b0 < B; b0 += frames_per_pass) {
    const int nb = std::min(frames_per_pass, B - b0);
    const float* l = (channels & kIn16)   // 16-bit host contract: the pointer walks 2-byte elements
        ? (const float*)((const uint16_t*)lidar + (size_t)b0 * px * (channels & ~kIn16))
        : lidar + (size_t)b0 * px * channels;
    const uint8_t* m = mask ? mask + (size_t)b0 * px : nullptr;
    float* lg = logits ? logits + (size_t)b0 * px * num_classes : nullptr;
    float* pr = probs ? probs + (size_t)b0 * px * num_classes : nullptr;
    int32_t* pd = preds + (size_t)b0 * px;
    int rc = (precision == PCLS_F16) ? run_pass<__half>(l, channels, m, raw, mean5, std5, nb, lg, pr, pd, s, ev)
                                     : run_pass<__nv_bfloat16>(l, channels, m, raw, mean5, std5, nb, lg, pr, pd, s, ev);
    if (rc) return rc;
  }
  return PCLS_OK;
}

static int check_forward_args(const Net& n, const float* lidar, int channels, const double* mean5, const double* std5,
                              int B, const int32_t* preds) {
  PCLS_REQUIRE(n.finalized, "pcls_net_forward: call pcls_net_finalize first");
  PCLS_REQUIRE(B >= 0 && B <= n.max_batch, "pcls_net_forward: batch %d exceeds max_batch %d", B, n.max_batch);
  const bool raw = mean5 != nullptr;
  if (lidar == nullptr && channels == 0) {   // input already staged in the net's own buffers (pcls_net_input_buffers)
    PCLS_REQUIRE(B <= n.frames_per_pass, "pcls_net_forward: a staged input must fit one pass (%d frames)", n.frames_per_pass);
    PCLS_REQUIRE(B == 0 || preds != nullptr, "pcls_net_forward: preds must not be NULL");
    return PCLS_OK;
  }
  if (channels & kIn16) {
    PCLS_REQUIRE(!raw && ((channels & ~kIn16) == 6 || (channels & ~kIn16) == 8),
                 "pcls_net_forward_in16: channels must be 6 or 8 (normalised 16-bit input), got %d", channels & ~kIn16);
    PCLS_REQUIRE(B == 0 || (lidar != nullptr && preds != nullptr), "pcls_net_forward_in16: lidar/preds must not be NULL");
    return PCLS_OK;
  }
  PCLS_REQUIRE(raw ? (channels == 5 || channels == 6) : channels == 6,
               "pcls_net_forward: channels must be 6 (normalised input) or 5/6 with mean/std (raw input), got %d", channels);
  PCLS_REQUIRE(!raw || std5 != nullptr, "pcls_net_forward: std is NULL");
  PCLS_REQUIRE(B == 0 || (lidar != nullptr && preds != nullptr), "pcls_net_forward: lidar/preds must not be NULL");
  return PCLS_OK;
}

int Net::forward(const float* lidar, int channels, const uint8_t* mask, const double* mean5, const double* std5, int B,
                 float* logits, float* probs, int32_t* preds, cudaStream_t s) {
  int rc = check_forward_args(*this, lidar, channels, mean5, std5, B, preds);
  if (rc) return rc;
  last_B = B;
  if (B == 0) return PCLS_OK;
  const bool raw = mean5 != nullptr;
  if (!use_graph) return run_all(lidar, channels, mask, raw, mean5, std5, B, logits, probs, preds, s, nullptr);

  // CUDA-graph replay: the whole forward (all passes) is captured once per distinct argument set on an internal
  // stream and replayed on the caller's stream; ~60-70 launches collapse into one graph launch.
  GraphKey key;
  memset(&key, 0, sizeof(key));
  key.lidar = lidar; key.mask = mask; key.logits = logits; key.probs = probs; key.preds = preds;
  key.channels = channels; key.B = B; key.raw = raw ? 1 : 0; key.conv_impl = conv_impl;
  for (int c = 0; c < 5; ++c) { key.norm[c] = raw ? mean5[c] : 0.0; key.norm[5 + c] = raw ? std5[c] : 0.0; }
  for (auto& g : graphs) {
    if (!memcmp(&g.key, &key, sizeof(key))) {
      g.stamp = ++graph_clock;
      graph_misses = 0;
      PCLS_CHECK_CUDA(cudaGraphLaunch(g.exec, s));
      return PCLS_OK;
    }
  }
  // A caller that hands in fresh buffers on every call (outputs kept alive, so the allocator cannot recycle them) would pay
  // a stream capture + cudaGraphInstantiate of ~60 nodes per forward: after a few misses in a row run the plain launches.
  if (++graph_misses > 4) return run_all(lidar, channels, mask, raw, mean5, std5, B, logits, probs, preds, s, nullptr);
  if (!cap_stream) PCLS_CHECK_CUDA(cudaStreamCreateWithFlags(&cap_stream, cudaStreamNonBlocking));
  PCLS_CHECK_CUDA(cudaStreamBeginCapture(cap_stream, cudaStreamCaptureModeRelaxed));
  rc = run_all(lidar, channels, mask, raw, mean5, std5, B, logits, probs, preds, cap_stream, nullptr);
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(cap_stream, &graph);
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (e != cudaSuccess) { set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e)); return PCLS_ERR_CUDA; }
  CachedGraph cg;
  cg.key = key;
  e = cudaGraphInstantiate(&cg.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); return PCLS_ERR_CUDA; }
  cg.stamp = ++graph_clock;
  if (graphs.size() >= 16) {  // evict the least recently used
    size_t victim = 0;
    for (size_t i = 1; i < graphs.size(); ++i) if (graphs[i].stamp < graphs[victim].stamp) victim = i;
    cudaGraphExecDestroy(graphs[victim].exec);
    graphs.erase(graphs.begin() + victim);
  }
  graphs.push_back(cg);
  PCLS_CHECK_CUDA(cudaGraphLaunch(cg.exec, s));
  return PCLS_OK;
}

void Net::drop_graphs() {
  for (auto& g : graphs) cudaGraphExecDestroy(g.exec);
  graphs.clear();
}

int Net::profile_ops(const float* lidar, int channels, const uint8_t* mask, const double* mean5, const double* std5,
                     int B, float* logits, float* probs, int32_t* preds, float* h_ms, cudaStream_t s) {
  int rc = check_forward_args(*this, lidar, channels, mean5, std5, B, preds);
  if (rc) return rc;
  PCLS_REQUIRE(B >= 1 && B <= frames_per_pass, "pcls_net_profile_ops: B must fit one pass (<= %d)", frames_per_pass);
  PCLS_REQUIRE(h_ms != nullptr, "pcls_net_profile_ops: h_ms is NULL");
  const int n = (int)ops.size() + 2;
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) PCLS_CHECK_CUDA(cudaEventCreate(&e));
  rc = run_all(lidar, channels, mask, mean5 != nullptr, mean5, std5, B, logits, probs, preds, s, ev.data());
  if (rc == PCLS_OK) {
    cudaError_t e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { set_error("profile: %s", cudaGetErrorString(e)); rc = PCLS_ERR_CUDA; }
  }
  if (rc == PCLS_OK)
    for (int i = 0; i < n; ++i) cudaEventElapsedTime(&h_ms[i], ev[i], ev[i + 1]);
  for (auto& e : ev) cudaEventDestroy(e);
  return rc;
}

bool Net::head_is_fused() const {
  if (!fuse_head || conv_impl != 0) return false;
  for (const auto& L : convs)
    if (L.out == logits_tensor) return L.tc_ok && (W % 128 == 0 || L.hp != nullptr);
  return false;
}

int Net::op_info(int i, char* name, int* family, int64_t* flops, int64_t* bytes) const {
  const int n = (int)ops.size() + 2;
  PCLS_REQUIRE(i >= 0 && i < n, "pcls_net_op_info: op index %d out of range", i);
  const int64_t HW = (int64_t)H * W;
  int fam = 0;
  int64_t fl = 0, by = 0;
  char buf[64];
  if (i == 0) {
    snprintf(buf, sizeof(buf), "input_stage");
    by = HW * (5 * 4 + 16 + 1);
  } else if (i == n - 1) {
    // fused into the epilogue of the logits convolution: that op carries the probability / prediction / mask bytes
    snprintf(buf, sizeof(buf), head_is_fused() ? "head_softmax_argmax(fused)" : "head_softmax_argmax");
    by = head_is_fused() ? 0 : HW * ((int64_t)num_classes * 4 * 2 + 4 + 1);
  } else {
    const OpRef& op = ops[i - 1];
    if (op.type == OP_CONV) {
      const ConvLayer& L = convs[op.index];
      const ConvParams& p = L.p;
      const char* mode = p.mode == MODE_1x1 ? "conv1x1" : p.mode == MODE_3x3_S1 ? "conv3x3" : p.mode == MODE_3x3_S2 ? "conv3x3s2" : "deconv1x4s2";
      const int64_t cin = L.cin_logical, cout = L.cout_logical;   // algorithmic work: the layer's own channels, not the padding
      snprintf(buf, sizeof(buf), "%s_%dx%d_w%d", mode, (int)cin, (int)cout, p.Wout);
      const int64_t taps = p.mode == MODE_DECONV ? 2 : p.ntaps;  // 2 of the 4 taps hit each output column
      fl = 2 * (int64_t)H * p.Wout * cin * cout * taps;
      by = (int64_t)H * p.Win * cin * 2 + (int64_t)H * p.Wout * cout * (p.out_f32 ? 4 : 2) +
           (int64_t)p.ntaps * cin * cout * 2;
      // logits layer with the head in its epilogue: it writes probabilities (the same NC x 4 bytes) instead of logits,
      // plus the 4-byte prediction, and reads the mask byte
      if (L.out == logits_tensor && head_is_fused()) by += (int64_t)H * p.Wout * (4 + 1);
      if (conv_impl == 0 && L.pool_src >= 0) {   // max-pool fused in: the kernel reads the un-pooled tensor instead of the pooled one
        by += (int64_t)H * (tensors[L.pool_src].width - p.Win) * cin * 2;
        snprintf(buf, sizeof(buf), "pool+%s_%dx%d_w%d", mode, (int)cin, (int)cout, p.Wout);
      }
      if (L.skip_src >= 0) {   // the skip is computed from the network input: 16 bytes per pixel instead of the 64-channel tensor
        const ConvLayer& P = convs[L.skip_src];
        by += (int64_t)H * W * tensors[P.in].stride * 2 + (int64_t)P.cin_logical * P.cout_logical * 2;
        fl += 2 * (int64_t)H * W * P.cin_logical * P.cout_logical;
      } else if (L.res0 >= 0) {
        by += (int64_t)H * p.Wout * cout * 2;
      }
      if (L.res1 >= 0) by += (int64_t)H * p.Wout * cout * 2;
      fam = (conv_impl == 0 && L.tc_ok) ? 1 : 0;
      if (L.skip_into >= 0) {                                 // runs inside the conv that reads its output
        snprintf(buf, sizeof(buf), "%s_%dx%d_w%d(fused)", mode, (int)cin, (int)cout, p.Wout);
        fl = 0; by = 0; fam = 0;
      }
      if (conv_impl == 0 && L.fused_into_up >= 0) {          // runs inside the transposed conv behind it
        snprintf(buf, sizeof(buf), "%s_%dx%d_w%d(fused)", mode, (int)cin, (int)cout, p.Wout);
        fl = 0; by = 0; fam = 0;
      }
      if (conv_impl == 0 && L.up_squeeze >= 0) {             // squeeze input -> up-sampled output, the squeeze tensor stays on chip
        const ConvLayer& Q = convs[L.up_squeeze];
        snprintf(buf, sizeof(buf), "conv1x1_%dx%d+%s_w%d", Q.cin_logical, Q.cout_logical, mode, p.Wout);
        fl += 2 * (int64_t)H * p.Win * Q.cin_logical * Q.cout_logical;
        by = (int64_t)H * p.Win * Q.cin_logical * 2 + (int64_t)H * p.Wout * cout * 2 +
             ((int64_t)Q.cin_logical * Q.cout_logical + (int64_t)p.ntaps * cin * cout) * 2;
        fam = 0;
      }
    } else if (op.type == OP_POOL) {
      const PoolLayer& L = pools[op.index];
      const bool fused = conv_impl == 0 && L.fused_conv >= 0;
      snprintf(buf, sizeof(buf), fused ? "maxpool3x3s2_c%d_w%d(fused)" : "maxpool3x3s2_c%d_w%d", tensors[L.in].channels, tensors[L.out].width);
      by = fused ? 0 : (int64_t)H * (tensors[L.in].width + tensors[L.out].width) * tensors[L.in].channels * 2;
    } else {
      const CamLayer& L = cams[op.index];
      snprintf(buf, sizeof(buf), "cam_c%d_w%d", L.C, tensors[L.in].width);
      fl = 2 * (int64_t)H * tensors[L.in].width * L.C * L.R * 2;
      by = (int64_t)H * tensors[L.in].width * L.C * 2 * 2;
    }
  }
  if (name) { strncpy(name, buf, 63); name[63] = 0; }
  if (family) *family = fam;
  if (flops) *flops = fl;
  if (bytes) *bytes = by;
  return PCLS_OK;
}

int Net::read_tensor(int t, int B, float* out, cudaStream_t s) {
  PCLS_REQUIRE(finalized && t >= 0 && t < (int)tensors.size(), "pcls_net_read_tensor: bad tensor id %d", t);
  PCLS_REQUIRE(B >= 0 && B <= frames_per_pass, "pcls_net_read_tensor: B exceeds the frames of one pass");
  PCLS_REQUIRE(t == 0 || tensors[t].first >= 0, "pcls_net_read_tensor: tensor %d is computed inside the conv that reads it "
               "(set keep_tensors or fuse_skip = 0 before finalize)", t);
  const TensorInfo& ti = tensors[t];
  const int64_t n = (int64_t)B * H * ti.width * ti.channels;
  if (ti.logits) { PCLS_CHECK_CUDA(cudaMemcpyAsync(out, tensor_ptr(t, B), n * 4, cudaMemcpyDeviceToDevice, s)); return PCLS_OK; }
  return precision == PCLS_F16 ? launch_tensor_to_f32<__half>((const __half*)tensor_ptr(t, B), out, n, ti.channels, ti.stride, s)
                               : launch_tensor_to_f32<__nv_bfloat16>((const __nv_bfloat16*)tensor_ptr(t, B), out, n, ti.channels, ti.stride, s);
}

Net::~Net() {
  drop_graphs();
  if (cap_stream) cudaStreamDestroy(cap_stream);
  if (arena) cudaFree(arena);
  if (weights) cudaFree(weights);
  tc_release();
}

}  // namespace pcls

using namespace pcls;

extern "C" int pcls_net_create(pcls_net** out, int H, int W, int precision, int max_batch) {
  PCLS_REQUIRE(out != nullptr, "pcls_net_create: out is NULL");
  PCLS_REQUIRE(H > 0 && W > 0 && max_batch > 0, "pcls_net_create: bad shape H=%d W=%d max_batch=%d", H, W, max_batch);
  PCLS_REQUIRE(precision == PCLS_F16 || precision == PCLS_BF16, "pcls_net_create: bad precision %d", precision);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("pcls_net_create: no CUDA device (libpclseg has no CPU fallback)");
    return PCLS_ERR_CUDA;
  }
  Net* n = new Net();
  n->H = H; n->W = W; n->precision = precision; n->max_batch = max_batch;
  n->add_tensor(W, 8, false);  // tensor 0: network input, 6 channels + 2 zero pad
  *out = reinterpret_cast<pcls_net*>(n);
  return PCLS_OK;
}

extern "C" void pcls_net_destroy(pcls_net* net) { delete reinterpret_cast<Net*>(net); }

extern "C" int pcls_net_tensor(pcls_net* net, int width, int channels, int is_logits) {
  Net* n = reinterpret_cast<Net*>(net);
  PCLS_REQUIRE(n != nullptr && !n->finalized, "pcls_net_tensor: bad or finalized net");
  PCLS_REQUIRE(width > 0 && channels > 0 && (is_logits || channels % 8 == 0),
               "pcls_net_tensor: width %d channels %d (activation channels must be a multiple of 8)", width, channels);
  return n->add_tensor(width, channels, is_logits != 0);
}

extern "C" int pcls_net_conv(pcls_net* net, const pcls_conv_desc* desc) {
  PCLS_REQUIRE(net != nullptr && desc != nullptr, "pcls_net_conv: NULL argument");
  return reinterpret_cast<Net*>(net)->add_conv(*desc);
}

extern "C" int pcls_net_maxpool3x3_s2(pcls_net* net, int in_tensor, int out_tensor) {
  PCLS_REQUIRE(net != nullptr, "pcls_net_maxpool3x3_s2: NULL net");
  return reinterpret_cast<Net*>(net)->add_pool(in_tensor, out_tensor);
}

extern "C" int pcls_net_cam(pcls_net* net, const pcls_cam_desc* desc) {
  PCLS_REQUIRE(net != nullptr && desc != nullptr, "pcls_net_cam: NULL argument");
  return reinterpret_cast<Net*>(net)->add_cam(*desc);
}

extern "C" int pcls_net_finalize(pcls_net* net, int logits_tensor, int num_classes, int none_index) {
  PCLS_REQUIRE(net != nullptr, "pcls_net_finalize: NULL net");
  return reinterpret_cast<Net*>(net)->finalize(logits_tensor, num_classes, none_index);
}

extern "C" int pcls_net_forward(pcls_net* net, const float* lidar, int channels, const uint8_t* mask,
                                const double* h_mean5, const double* h_std5, int B, float* logits, float* probs,
                                int32_t* preds, pcls_stream stream) {
  PCLS_REQUIRE(net != nullptr, "pcls_net_forward: NULL net");
  return reinterpret_cast<Net*>(net)->forward(lidar, channels, mask, h_mean5, h_std5, B, logits, probs, preds,
                                              (cudaStream_t)stream);
}

extern "C" int pcls_net_forward_in16(pcls_net* net, const void* lidar16, int channels, const uint8_t* mask, int B,
                                     float* logits, float* probs, int32_t* preds, pcls_stream stream) {
  PCLS_REQUIRE(net != nullptr, "pcls_net_forward_in16: NULL net");
  PCLS_REQUIRE(channels == 6 || channels == 8, "pcls_net_forward_in16: channels must be 6 or 8, got %d", channels);
  PCLS_REQUIRE(B == 0 || lidar16 != nullptr, "pcls_net_forward_in16: lidar16 is NULL");
  return reinterpret_cast<Net*>(net)->forward((const float*)lidar16, channels | kIn16, mask, nullptr, nullptr, B, logits,
                                              probs, preds, (cudaStream_t)stream);
}

extern "C" int pcls_net_input_buffers(pcls_net* net, void** input8, uint8_t** mask, int* frames) {
  Net* n = reinterpret_cast<Net*>(net);
  PCLS_REQUIRE(n != nullptr && n->finalized, "pcls_net_input_buffers: net is NULL or not finalized");
  if (input8) *input8 = n->tensor_ptr(0, n->frames_per_pass);
  if (mask) *mask = (uint8_t*)n->arena + n->mask_offset * (size_t)n->frames_per_pass;
  if (frames) *frames = n->frames_per_pass;
  return PCLS_OK;
}

extern "C" int pcls_net_read_tensor(pcls_net* net, int tensor, int B, float* out, pcls_stream stream) {
  PCLS_REQUIRE(net != nullptr && out != nullptr, "pcls_net_read_tensor: NULL argument");
  return reinterpret_cast<Net*>(net)->read_tensor(tensor, B, out, (cudaStream_t)stream);
}

extern "C" int pcls_net_num_ops(const pcls_net* net) {
  const Net* n = reinterpret_cast<const Net*>(net);
  return n ? (int)n->ops.size() + 2 : 0;
}

extern "C" int pcls_net_profile_ops(pcls_net* net, const float* lidar, int channels, const uint8_t* mask,
                                    const double* h_mean5, const double* h_std5, int B, float* logits, float* probs,
                                    int32_t* preds, float* h_ms, pcls_stream stream) {
  PCLS_REQUIRE(net != nullptr, "pcls_net_profile_ops: NULL net");
  return reinterpret_cast<Net*>(net)->profile_ops(lidar, channels, mask, h_mean5, h_std5, B, logits, probs, preds, h_ms,
                                                  (cudaStream_t)stream);
}

extern "C" int pcls_net_op_info(const pcls_net* net, int i, char* h_name, int* family, int64_t* flops_per_frame,
                                int64_t* bytes_per_frame) {
  PCLS_REQUIRE(net != nullptr, "pcls_net_op_info: NULL net");
  return reinterpret_cast<const Net*>(net)->op_info(i, h_name, family, flops_per_frame, bytes_per_frame);
}

extern "C" int pcls_net_launches_per_forward(const pcls_net* net) {
  const Net* n = reinterpret_cast<const Net*>(net);
  if (!n) return 0;
  // kernels one pass really launches: the input kernel, every op that is not folded into a neighbour (squeeze convs
  // computed by the transposed conv behind them, max-pools computed by the 1x1 conv behind them), and the standalone
  // head kernel unless the logits layer runs it in its epilogue
  int launches = 1;
  for (const OpRef& op : n->ops) {
    if (op.type == OP_CONV && n->conv_impl == 0 && n->convs[op.index].fused_into_up >= 0) continue;
    if (op.type == OP_CONV && n->convs[op.index].skip_into >= 0) continue;
    if (op.type == OP_POOL && n->conv_impl == 0 && n->pools[op.index].fused_conv >= 0) continue;
    ++launches;
  }
  return launches + (n->head_is_fused() ? 0 : 1);
}

extern "C" int64_t pcls_net_workspace_bytes(const pcls_net* net) {
  const Net* n = reinterpret_cast<const Net*>(net);
  return n ? (int64_t)(n->arena_bytes + n->weight_bytes) : 0;
}

extern "C" int pcls_net_set_option(pcls_net* net, const char* name, int value) {
  Net* n = reinterpret_cast<Net*>(net);
  PCLS_REQUIRE(n != nullptr && name != nullptr, "pcls_net_set_option: NULL argument");
  if (!strcmp(name, "conv_impl")) {
    PCLS_REQUIRE(value == 0 || value == 1, "conv_impl must be 0 or 1");
    bool skip_fused = false;   // (the fused skip tensor is never allocated: the CUDA-core path could not write it)
    for (const auto& L : n->convs) skip_fused = skip_fused || L.skip_into >= 0;
    PCLS_REQUIRE(value == 0 || !skip_fused, "conv_impl = 1 needs a net finalized with fuse_skip = 0 (or conv_impl = 1 set before)");
    n->conv_impl = value; return PCLS_OK;
  }
  if (!strcmp(name, "use_graph")) { n->use_graph = value != 0; if (!n->use_graph) n->drop_graphs(); return PCLS_OK; }
  if (!strcmp(name, "micro_batch")) {
    PCLS_REQUIRE(!n->finalized, "micro_batch must be set before pcls_net_finalize");
    PCLS_REQUIRE(value >= 0, "micro_batch must be >= 0");
    n->micro_batch = value; return PCLS_OK;
  }
  if (!strcmp(name, "keep_tensors")) {
    PCLS_REQUIRE(!n->finalized, "keep_tensors must be set before pcls_net_finalize");
    n->keep_tensors = value != 0; return PCLS_OK;
  }
  if (!strcmp(name, "tc_head")) { tc_head_mode = value; return PCLS_OK; }
  if (!strcmp(name, "cam_px")) { PCLS_REQUIRE(value >= 0 && value <= 2, "cam_px must be 0 (default), 1 or 2"); n->cam_px = value; n->drop_graphs(); return PCLS_OK; }
  if (!strcmp(name, "tc_nsplit")) { tc_nsplit_mode = value; return PCLS_OK; }
  if (!strcmp(name, "pad48")) {
    PCLS_REQUIRE(n->convs.empty(), "pad48 must be set before the first pcls_net_conv");
    pad48_mode = value; return PCLS_OK;
  }
  if (!strcmp(name, "pair_s2")) {
    PCLS_REQUIRE(n->convs.empty(), "pair_s2 must be set before the first pcls_net_conv");
    pair_s2_mode = value; return PCLS_OK;
  }
  if (!strcmp(name, "tc_halo")) { tc_halo_mode = value; return PCLS_OK; }
  if (!strcmp(name, "tc_rtma")) { tc_rtma_mode = value; n->drop_graphs(); return PCLS_OK; }
  if (!strcmp(name, "tc_tma_store")) { tc_tma_store_mode = value; return PCLS_OK; }
  if (!strcmp(name, "tc_group")) { tc_group_mode = value; return PCLS_OK; }
  if (!strcmp(name, "tc_res_tma")) { tc_res_tma_mode = value; return PCLS_OK; }
  if (!strcmp(name, "tc_split")) { tc_split_mode = value; return PCLS_OK; }
  if (!strcmp(name, "tc_vstream")) { tc_vstream_mode = value; return PCLS_OK; }
  if (!strcmp(name, "fuse_up")) {
    PCLS_REQUIRE(!n->finalized, "fuse_up must be set before pcls_net_finalize");
    n->fuse_up = value != 0; return PCLS_OK;
  }
  if (!strcmp(name, "fuse_pool")) {
    PCLS_REQUIRE(!n->finalized, "fuse_pool must be set before pcls_net_finalize");
    n->fuse_pool = value != 0; return PCLS_OK;
  }
  if (!strcmp(name, "fuse_skip")) {
    PCLS_REQUIRE(!n->finalized, "fuse_skip must be set before pcls_net_finalize");
    n->fuse_skip = value != 0; return PCLS_OK;
  }
  if (!strcmp(name, "fuse_head")) { n->fuse_head = value != 0; n->drop_graphs(); return PCLS_OK; }
  if (!strcmp(name, "tc_debug")) {  // per-role wait-cycle counters of conv_tc_kernel (development aid)
    PCLS_REQUIRE(!value || tc_debug_compiled, "tc_debug needs a library built with PCLS_NVCC_FLAGS=-DPCLS_TC_DEBUG=1");
    if (value && !tc_debug_buf) { PCLS_CHECK_CUDA(cudaMalloc(&tc_debug_buf, 148 * 24 * 8)); PCLS_CHECK_CUDA(cudaMemset(tc_debug_buf, 0, 148 * 24 * 8)); }
    if (!value && tc_debug_buf) { cudaFree(tc_debug_buf); tc_debug_buf = nullptr; }
    return PCLS_OK;
  }
  if (!strcmp(name, "tc_resident")) { tc_resident_mode = value; return PCLS_OK; }
  if (!strcmp(name, "tc_base_offset")) { tc_base_offset_mode = value; return PCLS_OK; }
  set_error("pcls_net_set_option: unknown option '%s'", name);
  return PCLS_ERR_INVALID;
}
