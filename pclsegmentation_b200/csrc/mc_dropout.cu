// Monte-Carlo dropout (sm_100a): the in-network dropout op of the stochastic net (Gal & Ghahramani, ICML 2016; Kendall
// et al., Bayesian SegNet, 2015), and the per-pixel accumulate / finalize over T stochastic passes (mean probabilities,
// predictive entropy, mutual information).  No reference call site: the reference's Dropout layers only act in training.
// The rules are stated in include/pclseg.h and restated in numpy by oracle/mc_dropout.py.
//
// dropout_kernel<T>: in place, one 16-byte vector (8 elements) and one Philox4x32-10 call per thread step, grid-stride
//   over the pass.  Integer work (Philox: 20 32-bit multiplies and ~40 xor / add per vector) and one float32 multiply per
//   kept element; 32 B of HBM traffic per vector.  The (seed, frame_base, pass) state is read from device memory after
//   pdl_wait(), so one captured CUDA graph serves every pass; the pass offset b0 of a micro-batched forward is a kernel
//   argument (known at capture).
// mc_accumulate_kernel / mc_finalize_kernel: one warp per 32 pixels; the NC x 32 probabilities are staged through shared
//   memory (coalesced loads, as head_kernel), lane = pixel for the per-pixel reductions.
#include "nn_kernels.cuh"

#include <math.h>

namespace pcls {

constexpr int MC_MAX_NC = 32;
constexpr int MC_WARPS = 8;
constexpr int MC_MAX_PASSES = 65536;

// Philox4x32-10 (Salmon et al., SC 2011): counter c, key k.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
  }
  return c;
}

template <typename T>
__global__ void __launch_bounds__(256)
dropout_kernel(int4* __restrict__ data, uint32_t n_vec, uint32_t vec_per_frame, uint32_t site, uint32_t thr, float scale,
               const DropState* __restrict__ state, uint32_t b0, int pdl_early) {
  pdl_trigger(pdl_early);
  pdl_wait();   // the tensor and the state are written by kernels in front of this one
  const unsigned long long seed = state->seed, frame_base = state->frame_base;
  const uint32_t ck = site | (state->pass << 16);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < n_vec; v += stride) {
    const uint32_t fl = v / vec_per_frame, g = v - fl * vec_per_frame;
    const unsigned long long f = frame_base + b0 + fl;
    const uint4 r = philox4x32_10(make_uint4(g, ck, (uint32_t)f, (uint32_t)(f >> 32)), key);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    int4 q = data[v];
    T* h = reinterpret_cast<T*>(&q);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t u0 = w[i] & 0xFFFFu, u1 = w[i] >> 16;   // element 8g + 2i, element 8g + 2i + 1
      h[2 * i] = u0 >= thr ? from_f32<T>(__fmul_rn(to_f32<T>(h[2 * i]), scale)) : from_f32<T>(0.0f);
      h[2 * i + 1] = u1 >= thr ? from_f32<T>(__fmul_rn(to_f32<T>(h[2 * i + 1]), scale)) : from_f32<T>(0.0f);
    }
    data[v] = q;
  }
}

__global__ void set_dropout_kernel(DropState* state, unsigned long long seed, unsigned long long frame_base,
                                   unsigned pass) {
  state->seed = seed;
  state->frame_base = frame_base;
  state->pass = pass;
}

__global__ void __launch_bounds__(MC_WARPS * 32)
mc_accumulate_kernel(const float* __restrict__ probs, int64_t n, int nc, int pass, float* __restrict__ acc_probs,
                     double* __restrict__ acc_entropy) {
  __shared__ float tile[MC_WARPS][32 * (MC_MAX_NC + 1)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* t = tile[warp];
  const int pitch = nc + 1;
  const float log_nc = logf((float)nc);
  const int64_t n_groups = (n + 31) / 32;
  for (int64_t g = (int64_t)blockIdx.x * MC_WARPS + warp; g < n_groups; g += (int64_t)gridDim.x * MC_WARPS) {
    const int64_t p0 = g * 32;
    const int np = n - p0 >= 32 ? 32 : (int)(n - p0);
    const int n_el = np * nc;
    const float* s = probs + p0 * nc;
    float* a = acc_probs + p0 * nc;
    for (int e = lane; e < n_el; e += 32) {
      const float p = __ldg(s + e);
      t[(e / nc) * pitch + (e % nc)] = p;
      a[e] = pass == 0 ? p : __fadd_rn(a[e], p);
    }
    __syncwarp();
    if (lane < np) {
      float v[MC_MAX_NC];
#pragma unroll
      for (int c = 0; c < MC_MAX_NC; ++c) v[c] = (c < nc) ? t[lane * pitch + c] : 0.0f;
      const double h = (double)normalised_entropy<MC_MAX_NC>(v, nc, log_nc);
      acc_entropy[p0 + lane] = pass == 0 ? h : acc_entropy[p0 + lane] + h;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(MC_WARPS * 32)
mc_finalize_kernel(const float* __restrict__ acc_probs, const double* __restrict__ acc_entropy,
                   const uint8_t* __restrict__ mask, int64_t n, int nc, int none_index, int n_passes,
                   float* __restrict__ out_probs, int32_t* __restrict__ out_preds, float* __restrict__ out_conf,
                   float* __restrict__ out_entropy, float* __restrict__ out_mi) {
  __shared__ float tile[MC_WARPS][32 * (MC_MAX_NC + 1)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* t = tile[warp];
  const int pitch = nc + 1;
  const float log_nc = logf((float)nc);
  const float tf = (float)n_passes;
  const int64_t n_groups = (n + 31) / 32;
  for (int64_t g = (int64_t)blockIdx.x * MC_WARPS + warp; g < n_groups; g += (int64_t)gridDim.x * MC_WARPS) {
    const int64_t p0 = g * 32;
    const int np = n - p0 >= 32 ? 32 : (int)(n - p0);
    const int n_el = np * nc;
    const float* s = acc_probs + p0 * nc;
    for (int e = lane; e < n_el; e += 32) t[(e / nc) * pitch + (e % nc)] = __ldg(s + e);
    __syncwarp();
    if (lane < np) {
      // (the float64 division before the class loop: its slow path is a call, made while no class value is live)
      const float EH = (out_entropy != nullptr || out_mi != nullptr)
                           ? (float)(acc_entropy[p0 + lane] / (double)n_passes) : 0.0f;
      float v[MC_MAX_NC];
      int best = 0;
      float bp = -1.0f;
#pragma unroll
      for (int c = 0; c < MC_MAX_NC; ++c) {
        v[c] = (c < nc) ? __fdiv_rn(t[lane * pitch + c], tf) : 0.0f;
        if (c < nc && v[c] > bp) { bp = v[c]; best = c; }   // first index on ties, as the head
      }
      const bool valid = mask == nullptr || mask[p0 + lane] != 0;
      if (out_preds != nullptr) out_preds[p0 + lane] = valid ? best : none_index;
      if (out_conf != nullptr) out_conf[p0 + lane] = valid ? bp : 0.0f;
      if (out_entropy != nullptr || out_mi != nullptr) {
        const float H = normalised_entropy<MC_MAX_NC>(v, nc, log_nc);
        if (out_entropy != nullptr) out_entropy[p0 + lane] = valid ? H : 0.0f;
        if (out_mi != nullptr) out_mi[p0 + lane] = valid ? fmaxf(0.0f, __fsub_rn(H, EH)) : 0.0f;
      }
      if (out_probs != nullptr) {
#pragma unroll
        for (int c = 0; c < MC_MAX_NC; ++c) if (c < nc) t[lane * pitch + c] = v[c];
      }
    }
    __syncwarp();
    if (out_probs != nullptr) {
      float* dst = out_probs + p0 * nc;
      for (int e = lane; e < n_el; e += 32) dst[e] = t[(e / nc) * pitch + (e % nc)];
    }
    __syncwarp();
  }
}

static int mc_grid(int64_t blocks, int per_sm) {
  const int64_t cap = (int64_t)sm_count() * per_sm;
  return (int)std::max<int64_t>(1, std::min(blocks, cap));
}

template <typename T>
int launch_dropout(void* data, int64_t n_vec, int64_t vec_per_frame, int site, uint32_t thr, float scale,
                   const DropState* state, int b0, cudaStream_t s) {
  if (n_vec == 0) return PCLS_OK;
  PCLS_REQUIRE(n_vec < (1ll << 31) && vec_per_frame > 0, "dropout: %lld vectors per pass exceed 2^31", (long long)n_vec);
  const int grid = mc_grid(ceil_div(n_vec, 256), 8);
  PCLS_CHECK_CUDA(launch_pdl(dropout_kernel<T>, dim3(grid), dim3(256), 0, s, (int4*)data, (uint32_t)n_vec,
                             (uint32_t)vec_per_frame, (uint32_t)site, thr, scale, state, (uint32_t)b0, pdl_early_now));
  return check_launch("dropout_kernel");
}
template int launch_dropout<__half>(void*, int64_t, int64_t, int, uint32_t, float, const DropState*, int, cudaStream_t);
template int launch_dropout<__nv_bfloat16>(void*, int64_t, int64_t, int, uint32_t, float, const DropState*, int,
                                           cudaStream_t);

int launch_set_dropout(DropState* state, unsigned long long seed, unsigned long long frame_base, unsigned pass,
                       cudaStream_t s) {
  set_dropout_kernel<<<1, 1, 0, s>>>(state, seed, frame_base, pass);
  return check_launch("set_dropout_kernel");
}

}  // namespace pcls

using namespace pcls;

extern "C" int pcls_mc_accumulate(const float* probs, int64_t n, int num_classes, int pass, float* acc_probs,
                                  double* acc_entropy, pcls_stream stream) {
  PCLS_REQUIRE(n >= 0, "pcls_mc_accumulate: negative n");
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= MC_MAX_NC, "pcls_mc_accumulate: num_classes %d not in [1,%d]",
               num_classes, MC_MAX_NC);
  PCLS_REQUIRE(pass >= 0 && pass < MC_MAX_PASSES, "pcls_mc_accumulate: pass %d not in [0,%d)", pass, MC_MAX_PASSES);
  PCLS_REQUIRE(n == 0 || (probs != nullptr && acc_probs != nullptr && acc_entropy != nullptr),
               "pcls_mc_accumulate: probs / acc_probs / acc_entropy must not be NULL");
  if (n == 0) return PCLS_OK;
  const int grid = mc_grid(ceil_div(ceil_div(n, 32), MC_WARPS), 8);
  mc_accumulate_kernel<<<grid, MC_WARPS * 32, 0, (cudaStream_t)stream>>>(probs, n, num_classes, pass, acc_probs,
                                                                          acc_entropy);
  return check_launch("mc_accumulate_kernel");
}

extern "C" int pcls_mc_finalize(const float* acc_probs, const double* acc_entropy, const uint8_t* mask, int64_t n,
                                int num_classes, int none_index, int n_passes, float* out_probs, int32_t* out_preds,
                                float* out_conf, float* out_entropy, float* out_mi, pcls_stream stream) {
  PCLS_REQUIRE(n >= 0, "pcls_mc_finalize: negative n");
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= MC_MAX_NC, "pcls_mc_finalize: num_classes %d not in [1,%d]",
               num_classes, MC_MAX_NC);
  PCLS_REQUIRE(none_index >= 0 && none_index < num_classes, "pcls_mc_finalize: none_index %d not in [0,%d)", none_index,
               num_classes);
  PCLS_REQUIRE(n_passes >= 1 && n_passes <= MC_MAX_PASSES, "pcls_mc_finalize: n_passes %d not in [1,%d]", n_passes,
               MC_MAX_PASSES);
  PCLS_REQUIRE(out_probs != nullptr || out_preds != nullptr || out_conf != nullptr || out_entropy != nullptr ||
                   out_mi != nullptr,
               "pcls_mc_finalize: no output given (out_probs / out_preds / out_conf / out_entropy / out_mi are all NULL)");
  PCLS_REQUIRE(n == 0 || (acc_probs != nullptr && acc_entropy != nullptr),
               "pcls_mc_finalize: acc_probs / acc_entropy must not be NULL");
  if (n == 0) return PCLS_OK;
  const int grid = mc_grid(ceil_div(ceil_div(n, 32), MC_WARPS), 8);
  mc_finalize_kernel<<<grid, MC_WARPS * 32, 0, (cudaStream_t)stream>>>(acc_probs, acc_entropy, mask, n, num_classes,
                                                                        none_index, n_passes, out_probs, out_preds,
                                                                        out_conf, out_entropy, out_mi);
  return check_launch("mc_finalize_kernel");
}
