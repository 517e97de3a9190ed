// Launchers of the network kernels (internal to libpclseg).
#pragma once
#include "common.cuh"

namespace pcls {

// Geometry of one convolution-like op as "taps": output pixel (h, wo) reads, for tap t, the input pixel
// (h + dh[t], wo * w_mul + dw[t]) when parity[t] < 0 or parity[t] == (wo & 1); transposed convs use
// w_shift: input column = (wo + dw[t]) >> 1.
enum ConvMode { MODE_1x1 = 0, MODE_3x3_S1 = 1, MODE_3x3_S2 = 2, MODE_DECONV = 3,
                MODE_PAIR6 = 4 /* tensor-core only: 3x3 s[1,2] on the pixel-pair view, taps (dh, dw in {0,1}) */,
                MODE_ROW3 = 5 /* tensor-core only: 1x3 conv (taps dw = -1,0,+1); the transposed conv with both output
                                 parities as N = 2 Cout */ };

struct ConvParams {
  int mode;
  int H, Win, Wout;
  int cin;            // logical input channels actually contracted (weights are zero beyond)
  int cin_pad;        // packed weight inner dim (multiple of 16)
  int in_channels;    // channel count (pixel stride) of the input tensor
  int cout;           // logical output channels
  int cout_pad;       // packed weight rows (multiple of 16)
  int out_channels;   // pixel stride of the output tensor
  int out_coff;       // channel offset of the write (tf.concat)
  int pad_left;       // MODE_3x3_S2: TF SAME left padding (0 for even Win)
  int act;
  int ntaps;          // 1, 9, 9, 4
  const void* in;     // T [B,H,Win,in_channels]
  void* out;          // T [B,H,Wout,out_channels]  or float [B,H,Wout,out_channels] when out_f32
  int out_f32;
  const void* res0;   // T, same geometry as out (pixel stride res0_channels), read at out_coff
  const void* res1;
  int res0_channels, res1_channels;
  const void* w;      // T packed [ntaps][cout_pad][cin_pad]
  const float* bias;  // [cout_pad]
};

template <typename T> int launch_conv_direct(const ConvParams& p, int B, cudaStream_t s);
template <typename T> int launch_net_input(const float* lidar, int channels, const uint8_t* mask_in, bool raw,
                                           const double* mean5, const double* std5, int64_t n_pixels, T* out8,
                                           uint8_t* mask_out, cudaStream_t s);
int launch_net_input16(const void* lidar16, int channels, const uint8_t* mask_in, int64_t n_pixels, void* out8,
                       uint8_t* mask_out, cudaStream_t s);
template <typename T> int launch_maxpool3x3_s2(const T* in, T* out, int B, int H, int Win, int Wout, int C,
                                               int pad_left, cudaStream_t s);

// max-pool 3x3 / s[1,2] fused with the 1x1 conv that consumes it (pool_conv.cu)
struct PoolConvParams {
  const void* in;      // T [B,H,Win,C]
  void* out;           // T [B,H,Wout,out_channels], channels [0,S) written
  const void* w;       // T [S][w_stride] folded 1x1 weights (K-major), channels >= C are not read
  const float* bias;   // [S]
  int H, Win, Wout, out_channels, w_stride, pad_left, act, n_strips, tiles_per_row;
  int zero_to;         // channels [S, zero_to) of the output are written as zeros (padded output tensors), 0: none
  int pdl_early;       // filled by the launcher (common.cuh)
};
bool pool_conv1x1_supported(int C, int S);
template <typename T> int launch_pool_conv1x1(const PoolConvParams& p, int C, int S, int B, cudaStream_t s);

// squeeze 1x1 conv fused with the transposed [1,4] / stride [1,2] conv that consumes it (squeeze_upconv.cu)
struct SqueezeUpconvParams {
  const void* in;      // T [B,H,W,C]
  void* out;           // T [B,H,2W,S]
  const void* w1;      // T [S][w1_stride] folded squeeze weights (K-major)
  const float* b1;     // [S]
  const void* w2;      // T [4][w2_cout_pad][w2_cin_pad] folded transposed-conv taps (out channel major, K-major rows)
  const float* b2;     // [S]
  int H, W, w1_stride, w2_cout_pad, w2_cin_pad, act1, act2;
  int rows, tiles_per_row;   // filled by the launcher
  int pdl_early;             // filled by the launcher (common.cuh)
};
bool squeeze_upconv_supported(int C, int S);
template <typename T> int launch_squeeze_upconv(const SqueezeUpconvParams& p, int C, int S, int B, cudaStream_t s);

struct CamParams {
  int C, R;            // channels, reduced channels (C / 16)
  const float* w1;     // [C][R]   folded squeeze weights
  const float* b1;     // [R]
  const float* w2;     // [R][C]   folded excitation weights
  const float* b2;     // [C]
  int pdl_early;       // filled by the launcher (common.cuh)
};
template <typename T> int launch_cam(const T* in, T* out, const CamParams& p, int B, int H, int W, cudaStream_t s);
template <typename T> int launch_tensor_to_f32(const T* in, float* out, int64_t n, int channels, int stride, cudaStream_t s);

int launch_head(const float* logits, const uint8_t* mask, int64_t n_pixels, int nc, int none_index, float* probs,
                int32_t* preds, cudaStream_t s);

// ---- segmentation head arithmetic ----
// Shared by the standalone head and the fused conv epilogues: softmax over v[0..nc), argmax over the
// rounded float32 probabilities (first index wins ties, like tf.argmax), mask fill.
template <int MAXNC>
__device__ __forceinline__ int softmax_argmax(float (&v)[MAXNC], int nc) {
  float m = v[0];
#pragma unroll
  for (int c = 1; c < MAXNC; ++c) if (c < nc) m = fmaxf(m, v[c]);
  float s = 0.0f;
#pragma unroll
  for (int c = 0; c < MAXNC; ++c) if (c < nc) { v[c] = expf(v[c] - m); s += v[c]; }
  int best = 0;
  float bp = -1.0f;
#pragma unroll
  for (int c = 0; c < MAXNC; ++c) if (c < nc) {
    v[c] = __fdiv_rn(v[c], s);
    if (v[c] > bp) { bp = v[c]; best = c; }
  }
  return best;
}

// Normalised entropy of probabilities v[0..nc): (-sum_c v_c * logf(v_c)) over the classes with v_c > 0, summed in class
// order in float32 with every product and sum rounded on its own, divided by log_nc = logf(nc); 0 when nc = 1.  Shared by
// pcls_confidence (calibration.cu) and the MC-dropout accumulate / finalize (mc_dropout.cu).
template <int MAXNC>
__device__ __forceinline__ float normalised_entropy(const float (&v)[MAXNC], int nc, float log_nc) {
  float h = 0.0f;
#pragma unroll
  for (int c = 0; c < MAXNC; ++c)
    if (c < nc && v[c] > 0.0f) h = __fadd_rn(h, __fmul_rn(v[c], logf(v[c])));
  return nc > 1 ? __fdiv_rn(-h, log_nc) : 0.0f;
}

// MC dropout (mc_dropout.cu): one in-place dropout op of the forward; `state` is the net's device-side
// (seed, frame_base, pass), written by pcls_net_set_dropout.  n_vec / vec_per_frame count 16-byte vectors.
struct DropState { unsigned long long seed, frame_base; unsigned int pass; };
template <typename T> int launch_dropout(void* data, int64_t n_vec, int64_t vec_per_frame, int site, uint32_t thr,
                                         float scale, const DropState* state, int b0, cudaStream_t s);
int launch_set_dropout(DropState* state, unsigned long long seed, unsigned long long frame_base, unsigned pass,
                       cudaStream_t s);

// 16-bit <-> float helpers
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == PCLS_ACT_RELU) return fmaxf(v, 0.0f);
  if (act == PCLS_ACT_LEAKY) return v > 0.0f ? v : 0.1f * v;
  return v;
}

// unpack / pack 8 x 16-bit values held in an int4
template <typename T> __device__ __forceinline__ void unpack8(const int4& q, float (&f)[8]) {
  const T* h = reinterpret_cast<const T*>(&q);
#pragma unroll
  for (int i = 0; i < 8; ++i) f[i] = to_f32<T>(h[i]);
}
template <typename T> __device__ __forceinline__ int4 pack8(const float (&f)[8]) {
  int4 q;
  T* h = reinterpret_cast<T*>(&q);
#pragma unroll
  for (int i = 0; i < 8; ++i) h[i] = from_f32<T>(f[i]);
  return q;
}

}  // namespace pcls
