// CUDA-core network kernels (sm_100a): generic direct convolution (every conv flavour of the two nets),
// network input conversion with the fused input stage, 3x3/s2 max-pool, the fused CAM gate.
//
// The direct convolution is the always-available CUDA path and the on-GPU cross-check for the tcgen05
// implicit-GEMM kernel (conv_tc.cu), which takes over every layer whose channel counts fit UMMA tiles.
#include "nn_kernels.cuh"

namespace pcls {

// --------------------------------------------------------------------------------------------------
// tap geometry shared by all conv implementations
// --------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool tap_source(const ConvParams& p, int tap, int h, int wo, int& hi, int& wi) {
  switch (p.mode) {
    case MODE_1x1:
      hi = h; wi = wo; return true;
    case MODE_3x3_S1:
      hi = h + tap / 3 - 1; wi = wo + tap % 3 - 1; break;
    case MODE_3x3_S2:  // TF SAME: total pad 1 for even Win -> 0 left / 1 right (SURVEY Appendix B)
      hi = h + tap / 3 - 1; wi = 2 * wo + tap % 3 - p.pad_left; break;
    default: {         // MODE_DECONV: out[m] += in[j] * w[k] with m = 2j + k - 1
      const int t = wo + 1 - tap;
      if (t < 0 || (t & 1)) return false;
      hi = h; wi = t >> 1; break;
    }
  }
  return hi >= 0 && hi < p.H && wi >= 0 && wi < p.Win;
}

// --------------------------------------------------------------------------------------------------
// direct convolution: 64 output pixels x 64 output channels per CTA, fp32 accumulate
// --------------------------------------------------------------------------------------------------
constexpr int DC_PX = 64, DC_CO = 64, DC_K = 16, DC_LD = 68;

template <typename T>
__global__ void __launch_bounds__(128)
conv_direct_kernel(const ConvParams p, const int64_t n_out) {
  __shared__ __align__(16) float As[DC_K][DC_LD];
  __shared__ __align__(16) float Ws[DC_K][DC_LD];
  const int tid = threadIdx.x;
  const int pxg = tid & 15, cg = tid >> 4;
  const int64_t pix0 = (int64_t)blockIdx.x * DC_PX;
  const int co0 = blockIdx.y * DC_CO;

  // the pixel / weight row this thread stages
  const int lpx = tid >> 1, lj = tid & 1;
  const int64_t lpix = pix0 + lpx;
  const bool lvalid = lpix < n_out;
  int lb = 0, lh = 0, lwo = 0;
  if (lvalid) {
    lwo = (int)(lpix % p.Wout);
    const int64_t r = lpix / p.Wout;
    lh = (int)(r % p.H);
    lb = (int)(r / p.H);
  }
  const int lco = co0 + lpx;  // weight row staged by this thread
  const T* in = reinterpret_cast<const T*>(p.in);
  const T* wt = reinterpret_cast<const T*>(p.w);

  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

  for (int tap = 0; tap < p.ntaps; ++tap) {
    int hi = 0, wi = 0;
    const bool src_ok = lvalid && tap_source(p, tap, lh, lwo, hi, wi);
    const T* src = in + (((int64_t)lb * p.H + hi) * p.Win + wi) * p.in_channels;
    const T* wrow = wt + ((int64_t)tap * p.cout_pad + lco) * p.cin_pad;
    for (int ck = 0; ck < p.cin_pad; ck += DC_K) {
      const int c = ck + 8 * lj;
      float f[8];
      if (src_ok && c < p.in_channels) {
        unpack8<T>(__ldg(reinterpret_cast<const int4*>(src + c)), f);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = 0.0f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) As[8 * lj + i][lpx] = f[i];
      if (lco < p.cout_pad) {
        unpack8<T>(__ldg(reinterpret_cast<const int4*>(wrow + c)), f);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = 0.0f;
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) Ws[8 * lj + i][lpx] = f[i];
      __syncthreads();
#pragma unroll
      for (int k = 0; k < DC_K; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(&As[k][pxg * 4]);
        const float4 w0 = *reinterpret_cast<const float4*>(&Ws[k][cg * 8]);
        const float4 w1 = *reinterpret_cast<const float4*>(&Ws[k][cg * 8 + 4]);
        const float av[4] = {a.x, a.y, a.z, a.w};
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
      }
      __syncthreads();
    }
  }

  // epilogue: bias (BN folded), activation, residual adds (after the activation), store
  const T* res0 = reinterpret_cast<const T*>(p.res0);
  const T* res1 = reinterpret_cast<const T*>(p.res1);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t pix = pix0 + pxg * 4 + i;
    if (pix >= n_out) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int co = co0 + cg * 8 + j;
      if (co >= p.cout) continue;
      float v = apply_act(acc[i][j] + __ldg(p.bias + co), p.act);
      if (res0) v += to_f32<T>(res0[pix * p.res0_channels + p.out_coff + co]);
      if (res1) v += to_f32<T>(res1[pix * p.res1_channels + p.out_coff + co]);
      if (p.out_f32) reinterpret_cast<float*>(p.out)[pix * p.out_channels + p.out_coff + co] = v;
      else reinterpret_cast<T*>(p.out)[pix * p.out_channels + p.out_coff + co] = from_f32<T>(v);
    }
  }
}

template <typename T>
int launch_conv_direct(const ConvParams& p, int B, cudaStream_t s) {
  const int64_t n_out = (int64_t)B * p.H * p.Wout;
  if (n_out == 0) return PCLS_OK;
  dim3 grid((unsigned)ceil_div(n_out, DC_PX), (unsigned)ceil_div(p.cout, DC_CO));
  conv_direct_kernel<T><<<grid, 128, 0, s>>>(p, n_out);
  return check_launch("conv_direct_kernel");
}
template int launch_conv_direct<__half>(const ConvParams&, int, cudaStream_t);
template int launch_conv_direct<__nv_bfloat16>(const ConvParams&, int, cudaStream_t);

// --------------------------------------------------------------------------------------------------
// network input: float32 [n,ch] -> 16-bit [n,8] (6 channels + 2 zero pad) + u8 mask, optional fused input stage
// --------------------------------------------------------------------------------------------------
struct Norm5f { double mean[5]; double std[5]; };

template <typename T>
__global__ void __launch_bounds__(256)
net_input_kernel(const float* __restrict__ lidar, int channels, const uint8_t* __restrict__ mask_in, int raw, Norm5f nrm,
                 int64_t n_pixels, T* __restrict__ out8, uint8_t* __restrict__ mask_out, int pdl_early) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  pdl_trigger(pdl_early);   // first kernel of the forward: tensor 0 / the mask buffer may still be read by the previous forward
  pdl_wait();
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pixels; p += stride) {
    const float* s = lidar + p * channels;
    float f[8];
#pragma unroll
    for (int c = 0; c < 5; ++c) f[c] = __ldg(s + c);
    bool m;
    if (raw) {  // inference.py:50-62 fused: mask = depth > 0, float64 normalise, zero where empty, append mask
      m = f[4] > 0.0f;
#pragma unroll
      for (int c = 0; c < 5; ++c) f[c] = m ? (float)(((double)f[c] - nrm.mean[c]) / nrm.std[c]) : 0.0f;
      f[5] = m ? 1.0f : 0.0f;
      if (mask_in) m = mask_in[p] != 0;
    } else {    // already normalised 6-channel reference input; channel 5 is the mask
      f[5] = __ldg(s + 5);
      // a derived mask follows channel 5 as tensor 0 stores it (16 bits, != +-0), like net_input16_kernel: a float32
      // value that rounds to a 16-bit zero (1e-8 in fp16) is an empty pixel in both, and NaN a valid one
      const T m5 = from_f32<T>(f[5]);
      m = mask_in ? (mask_in[p] != 0) : (*reinterpret_cast<const uint16_t*>(&m5) & 0x7FFFu) != 0;
    }
    f[6] = 0.0f; f[7] = 0.0f;
    reinterpret_cast<int4*>(out8)[p] = pack8<T>(f);
    mask_out[p] = m ? 1 : 0;
  }
}

template <typename T>
int launch_net_input(const float* lidar, int channels, const uint8_t* mask_in, bool raw, const double* mean5,
                     const double* std5, int64_t n_pixels, T* out8, uint8_t* mask_out, cudaStream_t s) {
  if (n_pixels == 0) return PCLS_OK;
  Norm5f nrm;
  for (int c = 0; c < 5; ++c) { nrm.mean[c] = raw ? mean5[c] : 0.0; nrm.std[c] = raw ? std5[c] : 1.0; }
  int64_t blocks = ceil_div(n_pixels, 256);
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  PCLS_CHECK_CUDA(launch_pdl(net_input_kernel<T>, dim3((unsigned)blocks), dim3(256), 0, s, lidar, channels, mask_in, raw ? 1 : 0, nrm,
                             n_pixels, out8, mask_out, pdl_early_now));
  return check_launch("net_input_kernel");
}
template int launch_net_input<__half>(const float*, int, const uint8_t*, bool, const double*, const double*, int64_t,
                                      __half*, uint8_t*, cudaStream_t);
template int launch_net_input<__nv_bfloat16>(const float*, int, const uint8_t*, bool, const double*, const double*,
                                             int64_t, __nv_bfloat16*, uint8_t*, cudaStream_t);

// 16-bit host contract (pcls_net_forward_in16): the normalised reference input already in the net's storage type,
// [.,6] (5 channels + mask channel, the reference's lidar_input layout) or [.,8] (tensor 0's own layout).  A pure
// re-pack: 12 / 16 B read, 16 + 1 B written per pixel, bit-identical to what net_input_kernel makes of the f32 input
// rounded to 16 bits.
__global__ void __launch_bounds__(256)
net_input16_kernel(const uint32_t* __restrict__ in, int channels, const uint8_t* __restrict__ mask_in, int64_t n_pixels,
                   int4* __restrict__ out8, uint8_t* __restrict__ mask_out, int pdl_early) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  pdl_trigger(pdl_early);
  pdl_wait();
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pixels; p += stride) {
    int4 v;
    if (channels == 8) {
      v = __ldg(reinterpret_cast<const int4*>(in) + p);
      v.w = 0;
    } else {
      const uint32_t* s = in + p * 3;
      v.x = (int)__ldg(s); v.y = (int)__ldg(s + 1); v.z = (int)__ldg(s + 2); v.w = 0;
    }
    const bool m = mask_in ? (mask_in[p] != 0) : (((uint32_t)v.z >> 16) & 0x7FFFu) != 0;   // channel 5 != +-0
    out8[p] = v;
    mask_out[p] = m ? 1 : 0;
  }
}

int launch_net_input16(const void* lidar16, int channels, const uint8_t* mask_in, int64_t n_pixels, void* out8,
                       uint8_t* mask_out, cudaStream_t s) {
  if (n_pixels == 0) return PCLS_OK;
  int64_t blocks = ceil_div(n_pixels, 256);
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  PCLS_CHECK_CUDA(launch_pdl(net_input16_kernel, dim3((unsigned)blocks), dim3(256), 0, s, (const uint32_t*)lidar16, channels, mask_in,
                             n_pixels, (int4*)out8, mask_out, pdl_early_now));
  return check_launch("net_input16_kernel");
}

// --------------------------------------------------------------------------------------------------
// tf.nn.max_pool2d(ksize=3, strides=[1,2], padding='SAME'): rows h-1..h+1, cols 2wo-pl .. 2wo-pl+2
// one thread = one output pixel x 8 channels (128-bit loads/stores); padding never wins the max
// --------------------------------------------------------------------------------------------------
template <typename T> struct Vec2;
template <> struct Vec2<__half> { using type = __half2; };
template <> struct Vec2<__nv_bfloat16> { using type = __nv_bfloat162; };

template <typename T>
__device__ __forceinline__ int4 max8(const int4& a, const int4& b) {
  using V = typename Vec2<T>::type;
  int4 r;
  const V* x = reinterpret_cast<const V*>(&a);
  const V* y = reinterpret_cast<const V*>(&b);
  V* o = reinterpret_cast<V*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) o[i] = __hmax2(x[i], y[i]);
  return r;
}

template <typename T> __device__ __forceinline__ int4 neg_inf8();
template <> __device__ __forceinline__ int4 neg_inf8<__half>() { return make_int4(0xFC00FC00, 0xFC00FC00, 0xFC00FC00, 0xFC00FC00); }
template <> __device__ __forceinline__ int4 neg_inf8<__nv_bfloat16>() { return make_int4(0xFF80FF80, 0xFF80FF80, 0xFF80FF80, 0xFF80FF80); }

// Column-streaming form: a thread owns one output column x 8 channels of one frame and walks down the H rows.  Per
// input row it takes the horizontal 3-max (three 128-bit loads, two of them shared with the neighbour thread through
// L1) and keeps the last two row maxima in registers, so every input vector is requested 1.5x instead of 4.5x.
template <typename T>
__global__ void __launch_bounds__(256)
maxpool3x3_s2_kernel(const int4* __restrict__ in, int4* __restrict__ out, int64_t n_cols, int H, int Win, int Wout,
                     int CV, int pad_left, int rows_per_seg) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // (frame, wo, cv)
  if (i >= n_cols) return;
  // blockIdx.y = row segment: a column walk keeps only one row of loads (48 B) per thread in flight, so the grid must
  // offer ~2 x the SMs' thread capacity to cover the DRAM latency; segments pay two halo rows each
  const int h0 = blockIdx.y * rows_per_seg, h1 = min(H, h0 + rows_per_seg);
  const int cv = (int)(i % CV);
  const int wo = (int)((i / CV) % Wout);
  const int64_t b = i / ((int64_t)CV * Wout);
  const int4* img = in + b * H * Win * CV + cv;
  int4* oimg = out + (b * H * Wout + wo) * CV + cv;
  const int w_lo = 2 * wo - pad_left;
  const int4 NEG = neg_inf8<T>();
  auto hrow = [&](int h) -> int4 {
    if (h < 0 || h >= H) return NEG;
    const int4* row = img + (int64_t)h * Win * CV;
    int4 m = NEG;
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) {
      const int wi = w_lo + dx;
      if (wi >= 0 && wi < Win) m = max8<T>(m, __ldg(row + (int64_t)wi * CV));
    }
    return m;
  };
  int4 prev = hrow(h0 - 1), cur = hrow(h0), nxt = hrow(h0 + 1);
  for (int h = h0; h < h1; ++h) {
    const int4 nxt2 = (h + 1 < h1) ? hrow(h + 2) : NEG;   // two rows of loads in flight per thread
    oimg[(int64_t)h * Wout * CV] = max8<T>(max8<T>(prev, cur), nxt);
    prev = cur; cur = nxt; nxt = nxt2;
  }
}

template <typename T>
int launch_maxpool3x3_s2(const T* in, T* out, int B, int H, int Win, int Wout, int C, int pad_left, cudaStream_t s) {
  const int CV = C / 8;
  const int64_t n_cols = (int64_t)B * Wout * CV;
  if (n_cols == 0) return PCLS_OK;
  // row segments: enough threads for >= 2 full waves of 2048 threads per SM, at least 8 rows per segment
  int segs = (int)ceil_div((int64_t)sm_count() * 2048 * 2, n_cols);
  if (segs > H / 8) segs = H / 8;
  if (segs < 1) segs = 1;
  const int rows_per_seg = (int)ceil_div(H, segs);
  segs = (int)ceil_div(H, rows_per_seg);
  maxpool3x3_s2_kernel<T><<<dim3((unsigned)ceil_div(n_cols, 256), (unsigned)segs), 256, 0, s>>>(
      reinterpret_cast<const int4*>(in), reinterpret_cast<int4*>(out), n_cols, H, Win, Wout, CV, pad_left, rows_per_seg);
  return check_launch("maxpool3x3_s2_kernel");
}
template int launch_maxpool3x3_s2<__half>(const __half*, __half*, int, int, int, int, int, int, cudaStream_t);
template int launch_maxpool3x3_s2<__nv_bfloat16>(const __nv_bfloat16*, __nv_bfloat16*, int, int, int, int, int, int,
                                                 cudaStream_t);

// --------------------------------------------------------------------------------------------------
// CAM (nets/SqueezeSegV2.py:66-70), one row-streaming kernel:
//   pool = maxpool7x7_SAME(x); s = relu(W1^T pool + b1); e = sigmoid(W2^T s + b2); out = x * e
// A CTA (128 threads) owns a strip of TW columns of one frame and walks down the H rows; a thread owns two horizontally
// adjacent pixels x 8 channels of the strip.  Per iteration, ONE __syncthreads:
//   stage   input row r+3 travels global -> smem ring with cp.async (TW + 6 columns; -inf outside the image)
//   phase A horizontal 7-max of row r from the ring for both pixels (their windows share six of their seven columns: 8
//           loads for the pair); the last seven horizontal maxima stay in registers -> vertical 7-max = pooled row r-3,
//           still in registers.  They ARE the A fragment of the squeeze MMA (mma.sync m16n8k16, fp32 accumulate; the K
//           order is a free permutation of the channels, chosen so that lane (g, t) holds channels 8 cv .. 8 cv + 7,
//           cv = 4 cvg + t, of its first pixel in fragment row g and of its second in row g + 8).  A warp covers 16 pixels x
//           32 channels and leaves its partial sums in its own [TW][8] fp32 tile.
//   phase B (row r-4) sum of the C/32 partial tiles -> bias + ReLU -> A fragment of the excitation MMAs, whose N order is
//           permuted so that lane (g, t) receives exactly its own 8 channels (b2 rides along as two extra K rows, split
//           hi + lo); sigmoid on the SFU, gate x (16 bytes per pixel from the ring), two coalesced 16-byte global stores.
// HBM traffic: (TW + 6) / TW reads + 1 write of the tensor.  Weights live in registers as MMA B fragments.
// Two pixels per thread because the one-pixel form's busiest unit was the LSU data pipe (shared-memory wavefronts, 64 %),
// 7 of its LDS.128 per pixel going to the horizontal 7-max; the pair also carries its second pixel in fragment rows 8-15
// that were idle there: half the MMAs, address arithmetic and loop overhead per pixel.  Measured at batch 32: C = 64
// 0.138 vs 0.185 ms, C = 128 0.143 vs 0.189 ms (the one-pixel kernel has since been removed).
// --------------------------------------------------------------------------------------------------
template <typename T> __device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]);
template <> __device__ __forceinline__ void mma16816<__half>(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
template <> __device__ __forceinline__ void mma16816<__nv_bfloat16>(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
template <typename T> __device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  T h[2] = {from_f32<T>(lo), from_f32<T>(hi)};
  return *reinterpret_cast<uint32_t*>(h);
}
template <typename T> __device__ __forceinline__ float2 unpack2(uint32_t v) {
  const T* h = reinterpret_cast<const T*>(&v);
  return make_float2(to_f32<T>(h[0]), to_f32<T>(h[1]));
}
// sigmoid(e) = 0.5 + 0.5 tanh(e / 2) with ONE SFU op (tanh.approx.f32, max relative error 2^-11) instead of ex2 + rcp
// (0.137 -> 0.127 ms at C = 64, 0.143 -> 0.132 ms at C = 128); the factor 1/2 is folded into W2 / b2.  x * sigmoid =
// fma(x/2, t, x/2).
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr int CAM_DIST = 3;   // rows of loads in flight (5 measured no faster: the per-row dependency chain bounds CAM)
constexpr int CAM_CTAS = 3;   // resident CTAs per SM the register allocation targets (4: 128 registers, spills, 0.137 -> 0.256 ms)
template <int C> struct CamGeom {
  static constexpr int CV = C / 8;              // 16-byte vectors per pixel (8 or 16)
  static constexpr int TW = 256 / CV;           // columns per CTA (32 or 16)
  static constexpr int PITCH = C * 2 + 32;      // bytes per ring pixel; 2 PITCH = 64 mod 128: the (pixel, 4 vectors) reads
                                                // of a quarter warp (2 threads' pixels x 64 bytes) fall on disjoint banks.
                                                // (with a pitch of C * 2 + 64 every LDS.128 took two wavefronts, ncu
                                                // l1tex shared wavefronts 70 M vs 36 M ideal)
  static constexpr int ROWB = (TW + 6) * PITCH; // bytes per ring slot
  static constexpr int DIST = CAM_DIST, NB = DIST + 6;   // ring: rows r-5 .. r+DIST resident (DIST rows of loads in flight)
  static constexpr int SMEM = NB * ROWB + (2 * (CV / 4) + 1) * TW * 8 * 4;
};

template <typename T, int C>
__global__ void __launch_bounds__(128, CAM_CTAS)
cam2_kernel(const int4* __restrict__ in, int4* __restrict__ out, CamParams p, int H, int W, int rows_per_seg) {
  using G = CamGeom<C>;
  constexpr int CV = G::CV, TW = G::TW, PITCH = G::PITCH, ROWB = G::ROWB, NB = G::NB, DIST = G::DIST;
  constexpr int R = C / 16;                // reduced channels (4 or 8)
  constexpr int NSTG = (TW + 6) * CV;      // 16-byte copies per staged row
  constexpr int LPT = (NSTG + 127) / 128;
  constexpr int CVG = CV / 4;              // warps per pixel group (2 or 4)
  constexpr int STILE = TW * 8 * 4;        // bytes of one partial squeeze tile [TW][8] fp32
  extern __shared__ int4 cam_smem[];       // ring [NB][ROWB] | squeeze tiles [2][CVG][TW][8] fp32
  unsigned char* const ring = reinterpret_cast<unsigned char*>(cam_smem);
  unsigned char* const St = ring + NB * ROWB;

  const int w0 = blockIdx.x * TW;
  const int64_t b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int cvg = warp % CVG, pg = warp / CVG;
  const int c0 = pg * 16 + 2 * g, cv = cvg * 4 + t;      // this thread's pixels c0, c0 + 1 (columns of the strip) and channel vector
  const int4 NEG = neg_inf8<T>();
  const int64_t rowv = (int64_t)W * CV;                  // vectors per image row

  // ---- squeeze weights: B fragments of the two k-steps.  K slot (2t', 2t'+1 | +8) <-> channels 8 cv(t') + 4u + {0,1 | 2,3}
  uint32_t w1f[2][2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int ch = cv * 8 + 4 * u;
    auto w1 = [&](int k) { return g < R ? p.w1[(ch + k) * R + g] : 0.0f; };   // W1[channel][j = g]
    w1f[u][0] = pack2<T>(w1(0), w1(1));
    w1f[u][1] = pack2<T>(w1(2), w1(3));
  }
  // ---- excitation weights: N slot n of tile q <-> channel 8 (4 cvg + n / 2) + 2q + n % 2, so that the accumulator of
  // lane (g, t) (columns 2t, 2t+1) is channel pair q of its own vector.  The tanh form's 1/2 is folded into W2 and b2.
  constexpr float NL2E = 0.5f;
  uint32_t w2f[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int chn = (cvg * 4 + (g >> 1)) * 8 + 2 * q + (g & 1);
    auto w2 = [&](int j) { return j < R ? NL2E * p.w2[j * C + chn] : 0.0f; };  // W2[j = k][channel]
    w2f[q] = pack2<T>(w2(2 * t), w2(2 * t + 1));
  }
  // b2 rides in K rows 8 + 2q, 9 + 2q of tile q (hi + lo: fp32 accuracy), where A holds 1.0 for that tile only; the other
  // rows >= 8 meet zeros in A, so ONE register (lane t' holds the rows of tile q = t') serves all four tiles
  uint32_t w2b;
  {
    const float bias = NL2E * p.b2[(cvg * 4 + (g >> 1)) * 8 + 2 * t + (g & 1)];
    const float hi = to_f32<T>(from_f32<T>(bias));
    w2b = pack2<T>(hi, bias - hi);
  }
  const uint32_t one2 = pack2<T>(1.0f, 1.0f);

  // ---- staging: this thread's copies of a row (fixed columns, the source advances one image row per call) ----
  const int4* const fin = in + b * H * rowv;                 // this frame (CTA-uniform); per-thread offsets stay 32-bit
  int4* const fout = out + b * H * rowv;
  // copy k: column w0 - 3 + (tid + 128 k) / CV, vector tid % CV
  unsigned sptr = (unsigned)((w0 - 3 + (int)threadIdx.x / CV) * CV + threadIdx.x % CV);
  const unsigned soff = (unsigned)__cvta_generic_to_shared(ring) + (threadIdx.x / CV) * PITCH + (threadIdx.x % CV) * 16;
  bool sok[LPT];
#pragma unroll
  for (int k = 0; k < LPT; ++k) {
    const int i = threadIdx.x + k * 128;
    const int col = w0 - 3 + i / CV;
    sok[k] = i < NSTG && col >= 0 && col < W;
    if (i < NSTG && !sok[k])                                               // columns outside the image: -inf, written once
      for (int sl = 0; sl < NB; ++sl) *reinterpret_cast<int4*>(ring + sl * ROWB + (i / CV) * PITCH + (i % CV) * 16) = NEG;
  }
  const float b1x = 2 * t < R ? p.b1[2 * t] : 0.0f, b1y = 2 * t + 1 < R ? p.b1[2 * t + 1] : 0.0f;
  // blockIdx.z = row segment [h0, h1) of the strip (small batches: more CTAs than SMs; a segment re-reads three rows
  // above and below).  The walk starts at input row a0 = max(h0 - 3, 0).
  pdl_trigger(p.pdl_early);   // PDL (common.cuh): the weight fragments above are independent of the producing layer
  pdl_wait();
  const int h0 = blockIdx.z * rows_per_seg, h1 = min(H, h0 + rows_per_seg);
  const int a0 = h0 - 3 < 0 ? 0 : h0 - 3;
  sptr += (unsigned)a0 * (unsigned)rowv;
  auto stage_row = [&](int r, int slot) {
    if (r < H && r <= h1 + 2) {
#pragma unroll
      for (int k = 0; k < LPT; ++k)
        if (sok[k])
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(soff + k * (128 / CV) * PITCH + slot * ROWB),
                       "l"(fin + (unsigned)(sptr + k * 128)) : "memory");   // 32-bit wrap: sptr is "negative" left of the image
      sptr += (unsigned)rowv;
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  // ---- per-thread offsets ----
  const unsigned a_off = c0 * PITCH + cv * 16;            // ring: pixel c0 - 3 (+ d * PITCH), this vector
  const unsigned s_off = ((pg * 8 + g) * 4 + t) * 16;     // squeeze tile [pixel pair][t]: {c0: columns 2t, 2t+1 | c0 + 1: same} = one
                                                          // conflict-free 16-byte access per lane
  const bool ok0 = (w0 + c0) < W, ok1 = (w0 + c0 + 1) < W;
  unsigned optr = (unsigned)((w0 + c0) * CV + cv) + (unsigned)h0 * (unsigned)rowv;

  int4 win0[7], win1[7];   // horizontal maxima of the last seven input rows (slot = row mod 7)
#pragma unroll
  for (int k = 0; k < 7; ++k) { win0[k] = NEG; win1[k] = NEG; }

  for (int r = 0; r < DIST; ++r) stage_row(a0 + r, r);
  int sc = 0;                                             // ring slot of row r ((r - a0) mod NB)
  for (int r0 = a0; r0 < h1 + 4; r0 += 7) {
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const int r = r0 + j;
      if (r >= h1 + 4) break;
      stage_row(r + DIST, sc + DIST >= NB ? sc + DIST - NB : sc + DIST);
      asm volatile("cp.async.wait_group %0;" ::"n"(DIST) : "memory");    // row r has landed (this thread's copies)
      __syncthreads();

      // ---------------- phase A: pooled row r - 3 of both pixels, squeeze partial sums -> tiles [r & 1] ----------------
      if (r < h1 + 3) {
        int4 hm0 = NEG, hm1 = NEG;                                         // rows below the image pad with -inf
        if (r < H) {
          const unsigned char* src = ring + sc * ROWB + a_off;
          int4 m6 = *reinterpret_cast<const int4*>(src + PITCH);                     // columns shared by both windows
#pragma unroll
          for (int d = 2; d < 7; ++d) m6 = max8<T>(m6, *reinterpret_cast<const int4*>(src + d * PITCH));
          hm0 = max8<T>(m6, *reinterpret_cast<const int4*>(src));
          hm1 = max8<T>(m6, *reinterpret_cast<const int4*>(src + 7 * PITCH));
        }
        win0[j] = hm0; win1[j] = hm1;
        if (r >= h0 + 3) {
          int4 vm0 = win0[0], vm1 = win1[0];
#pragma unroll
          for (int k = 1; k < 7; ++k) { vm0 = max8<T>(vm0, win0[k]); vm1 = max8<T>(vm1, win1[k]); }
          // rows g / g + 8 of the fragment = pixels c0 / c0 + 1 (columns right of the image carry -inf: never stored)
          float sq[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          const uint32_t fa0[4] = {(uint32_t)vm0.x, (uint32_t)vm1.x, (uint32_t)vm0.y, (uint32_t)vm1.y};
          const uint32_t fa1[4] = {(uint32_t)vm0.z, (uint32_t)vm1.z, (uint32_t)vm0.w, (uint32_t)vm1.w};
          mma16816<T>(sq, fa0, w1f[0]);
          mma16816<T>(sq, fa1, w1f[1]);
          *reinterpret_cast<float4*>(St + ((r & 1) * CVG + cvg) * STILE + s_off) = make_float4(sq[0], sq[1], sq[2], sq[3]);
        }
      }

      // ---------------- phase B: gate and store row r - 4 (tiles [(r - 1) & 1]) ----------------
      if (r >= h0 + 4) {
        float2 sv0 = make_float2(b1x, b1y), sv1 = sv0;
#pragma unroll
        for (int k = 0; k < CVG; ++k) {
          const float4 pa = *reinterpret_cast<const float4*>(St + (((r - 1) & 1) * CVG + k) * STILE + s_off);
          sv0.x += pa.x; sv0.y += pa.y; sv1.x += pa.z; sv1.y += pa.w;
        }
        uint32_t sa[4] = {pack2<T>(fmaxf(sv0.x, 0.0f), fmaxf(sv0.y, 0.0f)), pack2<T>(fmaxf(sv1.x, 0.0f), fmaxf(sv1.y, 0.0f)), 0u, 0u};
        const int sb = sc + NB - 4 >= NB ? sc - 4 : sc + NB - 4;           // ring slot of input row r - 4
        const int4 xv0 = *reinterpret_cast<const int4*>(ring + sb * ROWB + a_off + 3 * PITCH);
        const int4 xv1 = *reinterpret_cast<const int4*>(ring + sb * ROWB + a_off + 4 * PITCH);
        const uint32_t xw0[4] = {(uint32_t)xv0.x, (uint32_t)xv0.y, (uint32_t)xv0.z, (uint32_t)xv0.w};
        const uint32_t xw1[4] = {(uint32_t)xv1.x, (uint32_t)xv1.y, (uint32_t)xv1.z, (uint32_t)xv1.w};
        uint32_t o0[4], o1[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float e[4] = {0.0f, 0.0f, 0.0f, 0.0f};
          const uint32_t bq[2] = {w2f[q], w2b};
          sa[2] = t == q ? one2 : 0u;
          sa[3] = sa[2];
          mma16816<T>(e, sa, bq);
          const float2 x0 = unpack2<T>(xw0[q]), x1 = unpack2<T>(xw1[q]);
          const float h0 = 0.5f * x0.x, h1 = 0.5f * x0.y, h2 = 0.5f * x1.x, h3 = 0.5f * x1.y;
          o0[q] = pack2<T>(fmaf(h0, tanh_approx(e[0]), h0), fmaf(h1, tanh_approx(e[1]), h1));
          o1[q] = pack2<T>(fmaf(h2, tanh_approx(e[2]), h2), fmaf(h3, tanh_approx(e[3]), h3));
        }
        if (ok0) fout[optr] = make_int4((int)o0[0], (int)o0[1], (int)o0[2], (int)o0[3]);
        if (ok1) fout[optr + CV] = make_int4((int)o1[0], (int)o1[1], (int)o1[2], (int)o1[3]);
        optr += (unsigned)rowv;
      }
      sc = sc + 1 == NB ? 0 : sc + 1;
    }
  }
}

template <typename T>
int launch_cam(const T* in, T* out, const CamParams& p, int B, int H, int W, cudaStream_t s) {
  if (B == 0) return PCLS_OK;
  PCLS_REQUIRE(p.C == 64 || p.C == 128, "CAM: channels must be 64 or 128, got %d", p.C);
  PCLS_REQUIRE(p.R == p.C / 16, "CAM: reduced channels must be C/16");
  const int TW = 256 / (p.C / 8);
  // row segments (>= 8 rows each): minimise  waves x iterations per CTA  with CAM_CTAS CTAs resident per SM; a segment of
  // n rows runs n + 7 iterations (three rows of halo above / below and the pipeline drain)
  const int64_t strips = ceil_div(W, TW) * (int64_t)B, slots = (int64_t)sm_count() * CAM_CTAS;
  int segs = 1;
  int64_t best = -1;
  for (int sgs = 1; sgs <= (H >= 8 ? H / 8 : 1); ++sgs) {
    const int64_t cost = ceil_div(strips * sgs, slots) * (ceil_div(H, sgs) + 7);
    if (best < 0 || cost < best) { best = cost; segs = sgs; }
  }
  const int rows_per_seg = (int)ceil_div(H, segs);
  segs = (int)ceil_div(H, rows_per_seg);
  dim3 grid((unsigned)ceil_div(W, TW), (unsigned)B, (unsigned)segs);
  const int smem = p.C == 64 ? CamGeom<64>::SMEM : CamGeom<128>::SMEM;
  auto kern = p.C == 64 ? cam2_kernel<T, 64> : cam2_kernel<T, 128>;
  static bool configured[64][2] = {};   // function attributes are per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (!configured[dev & 63][p.C == 128]) {
    PCLS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    PCLS_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    configured[dev & 63][p.C == 128] = true;
  }
  CamParams q = p;
  q.pdl_early = pdl_early_now;
  PCLS_CHECK_CUDA(launch_pdl(kern, grid, dim3(128), (size_t)smem, s, reinterpret_cast<const int4*>(in),
                             reinterpret_cast<int4*>(out), q, H, W, rows_per_seg));
  return check_launch("cam2_kernel");
}
template int launch_cam<__half>(const __half*, __half*, const CamParams&, int, int, int, cudaStream_t);
template int launch_cam<__nv_bfloat16>(const __nv_bfloat16*, __nv_bfloat16*, const CamParams&, int, int, int, cudaStream_t);

// --------------------------------------------------------------------------------------------------
// n dense output elements [pixels][channels]; the input holds `stride` >= channels values per pixel (padded tensors)
template <typename T>
__global__ void tensor_to_f32_kernel(const T* __restrict__ in, float* __restrict__ out, int64_t n, int channels, int stride) {
  const int64_t step = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step)
    out[i] = to_f32<T>(in[channels == stride ? i : (i / channels) * stride + i % channels]);
}
template <typename T>
int launch_tensor_to_f32(const T* in, float* out, int64_t n, int channels, int stride, cudaStream_t s) {
  if (n == 0) return PCLS_OK;
  int64_t blocks = ceil_div(n, 256);
  if (blocks > 65535) blocks = 65535;
  tensor_to_f32_kernel<T><<<(int)blocks, 256, 0, s>>>(in, out, n, channels, stride);
  return check_launch("tensor_to_f32_kernel");
}
template int launch_tensor_to_f32<__half>(const __half*, float*, int64_t, int, int, cudaStream_t);
template int launch_tensor_to_f32<__nv_bfloat16>(const __nv_bfloat16*, float*, int64_t, int, int, cudaStream_t);

}  // namespace pcls
