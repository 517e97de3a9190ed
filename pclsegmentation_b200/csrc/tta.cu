// Test-time augmentation (sm_100a): the mirrored / yaw-rotated views of raw range images as network input, and the
// merge of the views' probabilities back onto the source pixels (no reference call site: the reference trains with
// RANDOM_FLIPPING / SHIFT_LEFT_RIGHT but infers on one view).  The rules are stated in include/pclseg.h.
//
// tta_views_kernel<T>: one thread per source pixel reads the raw float32 pixel once (20 / 24 B) and writes the 16-byte
// network-input pixel and the mask byte of every view (T x 17 B).  A warp's 32 consecutive source columns land on 32
// consecutive view columns (reversed under the mirror, split in two at the roll's wrap point), so the 128-bit stores stay
// coalesced.
//
// tta_merge_kernel: one warp per 32 output pixels.  Per view it stages the 32 view pixels x NC probabilities through
// shared memory (coalesced loads, as head_kernel does), then lane = pixel adds them in view order.  Bytes per output
// pixel: T x NC x 4 + 1 read, 4 (+ NC x 4 with merged probabilities) written.
//
// Bit-exactness: the rotation is spelled with __dmul_rn / __dsub_rn / __dadd_rn and the merge with __fadd_rn /
// __fdiv_rn, so nvcc cannot contract them into FMAs and numpy reproduces every rounding (oracle/tta.py).
#include "nn_kernels.cuh"

#include <math.h>

namespace pcls {

constexpr int TTA_MAX_VIEWS = PCLS_TTA_MAX_VIEWS;
constexpr int TTA_MAX_NC = 32;
constexpr int TTA_WARPS = 8;
constexpr int TTA_LOADS = 8;   // merge: loads per lane issued before they are staged

struct TtaViews {
  int n;
  int flip[TTA_MAX_VIEWS], shift[TTA_MAX_VIEWS];
  double c[TTA_MAX_VIEWS], s[TTA_MAX_VIEWS];
};
struct TtaNorm { double mean[5], std[5]; };

// view column of source column w: the mirror first (w -> W-1-w), then the roll by shift
__device__ __forceinline__ int tta_column(const TtaViews& v, int t, int w, int W) {
  int c = v.flip[t] ? W - 1 - w : w;
  c += v.shift[t];
  return c >= W ? c - W : c;
}

template <typename T>
__global__ void __launch_bounds__(256)
tta_views_kernel(const float* __restrict__ raw, int channels, int B, int H, int W, TtaViews v, TtaNorm nrm,
                 int4* __restrict__ input8, uint8_t* __restrict__ mask) {
  const int64_t HW = (int64_t)H * W, n_pixels = (int64_t)B * HW;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pixels; p += stride) {
    const float* s = raw + p * channels;
    const float x = __ldg(s), y = __ldg(s + 1);
    const bool m = __ldg(s + 4) > 0.0f;
    // z, remission and range are the same in every view
    float f[8];
#pragma unroll
    for (int c = 2; c < 5; ++c) f[c] = m ? (float)(((double)__ldg(s + c) - nrm.mean[c]) / nrm.std[c]) : 0.0f;
    f[5] = m ? 1.0f : 0.0f;
    f[6] = f[7] = 0.0f;
    const int b = (int)(p / HW);
    const int64_t rem = p - (int64_t)b * HW;
    const int h = (int)(rem / W), w = (int)(rem - (int64_t)h * W);
    for (int t = 0; t < v.n; ++t) {
      const float yf = v.flip[t] ? -y : y;
      double xd = (double)x, yd = (double)yf;
      if (v.shift[t] != 0) {   // shift 0: no rotation at all, so signed zeros pass through as net_input_kernel sees them
        const double xr = __dsub_rn(__dmul_rn(v.c[t], xd), __dmul_rn(v.s[t], yd));
        const double yr = __dadd_rn(__dmul_rn(v.s[t], xd), __dmul_rn(v.c[t], yd));
        xd = xr; yd = yr;
      }
      f[0] = m ? (float)((xd - nrm.mean[0]) / nrm.std[0]) : 0.0f;
      f[1] = m ? (float)((yd - nrm.mean[1]) / nrm.std[1]) : 0.0f;
      const int64_t o = ((int64_t)t * B + b) * HW + (int64_t)h * W + tta_column(v, t, w, W);
      input8[o] = pack8<T>(f);
      mask[o] = m ? 1 : 0;
    }
  }
}

__global__ void __launch_bounds__(TTA_WARPS * 32)
tta_merge_kernel(const float* __restrict__ probs, const uint8_t* __restrict__ mask, int B, int H, int W, int nc,
                 int none_index, TtaViews v, float* __restrict__ out_probs, int32_t* __restrict__ out_preds) {
  __shared__ float tile[TTA_WARPS][32 * (TTA_MAX_NC + 1)];
  __shared__ int64_t vpix[TTA_WARPS][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* tl = tile[warp];
  int64_t* vp = vpix[warp];
  const int pitch = nc + 1;
  const int step_i = 32 / nc, step_c = 32 % nc;   // element e -> e + 32
  const int64_t HW = (int64_t)H * W, n_pixels = (int64_t)B * HW;
  const int64_t n_groups = (n_pixels + 31) / 32;
  for (int64_t g = (int64_t)blockIdx.x * TTA_WARPS + warp; g < n_groups; g += (int64_t)gridDim.x * TTA_WARPS) {
    const int64_t p0 = g * 32, p = p0 + lane;
    const int np = (int)min((int64_t)32, n_pixels - p0);
    const int b = (int)(p / HW);
    const int64_t rem = p - (int64_t)b * HW;
    const int h = (int)(rem / W), w = (int)(rem - (int64_t)h * W);
    float acc[TTA_MAX_NC];
    bool valid = false;
    const int n_el = np * nc;
    for (int i = 0; i < v.n; ++i) {
      const int t = i;                                      // views are summed in view order
      const int64_t q = ((int64_t)t * B + b) * HW + (int64_t)h * W + tta_column(v, t, w, W);   // this view's pixel
      if (t == 0 && lane < np) valid = mask[q] != 0;       // every view's mask is a permutation of the source mask
      vp[lane] = q;
      __syncwarp();
      // element e = lane + 32 k of the warp's np x nc block is (pixel ei, class ec), stepped without a division; the
      // loads of a batch are all issued before the first shared store, so TTA_LOADS of them are in flight per lane
      int ei = lane / nc, ec = lane - (lane / nc) * nc;
      for (int e0 = 0; e0 < n_el; e0 += 32 * TTA_LOADS) {
        float val[TTA_LOADS];
        int vi[TTA_LOADS], vc[TTA_LOADS];
#pragma unroll
        for (int k = 0; k < TTA_LOADS; ++k) {
          vi[k] = ei; vc[k] = ec;
          val[k] = e0 + 32 * k + lane < n_el ? __ldg(probs + vp[ei] * nc + ec) : 0.0f;
          ec += step_c; ei += step_i;
          if (ec >= nc) { ec -= nc; ++ei; }
        }
#pragma unroll
        for (int k = 0; k < TTA_LOADS; ++k)
          if (e0 + 32 * k + lane < n_el) tl[vi[k] * pitch + vc[k]] = val[k];
      }
      __syncwarp();
#pragma unroll
      for (int c = 0; c < TTA_MAX_NC; ++c)
        if (c < nc) acc[c] = i == 0 ? tl[lane * pitch + c] : __fadd_rn(acc[c], tl[lane * pitch + c]);
      __syncwarp();
    }
    if (lane < np) {
      const float tf = (float)v.n;
      int best = 0;
      float bp = -1.0f;
#pragma unroll
      for (int c = 0; c < TTA_MAX_NC; ++c) if (c < nc) {
        acc[c] = __fdiv_rn(acc[c], tf);
        if (acc[c] > bp) { bp = acc[c]; best = c; }   // first index on ties, as the head
      }
      out_preds[p] = valid ? best : none_index;
      if (out_probs != nullptr) {
#pragma unroll
        for (int c = 0; c < TTA_MAX_NC; ++c) if (c < nc) tl[lane * pitch + c] = acc[c];
      }
    }
    __syncwarp();
    if (out_probs != nullptr) {
      float* dst = out_probs + p0 * nc;
      int ei = lane / nc, ec = lane - (lane / nc) * nc;
      for (int e = lane; e < n_el; e += 32) {
        dst[e] = tl[ei * pitch + ec];
        ec += step_c; ei += step_i;
        if (ec >= nc) { ec -= nc; ++ei; }
      }
    }
    __syncwarp();
  }
}

// The checks both entry points share; fills `v` (cos / sin may be NULL for the merge).
static int tta_check_views(const char* who, int W, int n_views, const int* h_flip, const int* h_shift,
                           const double* h_cos, const double* h_sin, bool need_rotation, TtaViews& v) {
  PCLS_REQUIRE(n_views >= 1 && n_views <= TTA_MAX_VIEWS, "%s: n_views %d not in [1,%d]", who, n_views, TTA_MAX_VIEWS);
  PCLS_REQUIRE(h_flip != nullptr && h_shift != nullptr, "%s: h_flip / h_shift must not be NULL", who);
  PCLS_REQUIRE(!need_rotation || (h_cos != nullptr && h_sin != nullptr), "%s: h_cos / h_sin must not be NULL", who);
  v.n = n_views;
  for (int t = 0; t < n_views; ++t) {
    PCLS_REQUIRE(h_flip[t] == 0 || h_flip[t] == 1, "%s: view %d: flip %d is not 0 or 1", who, t, h_flip[t]);
    PCLS_REQUIRE(h_shift[t] >= 0 && h_shift[t] < W, "%s: view %d: shift %d not in [0,%d)", who, t, h_shift[t], W);
    for (int u = 0; u < t; ++u)
      PCLS_REQUIRE(h_flip[u] != h_flip[t] || h_shift[u] != h_shift[t], "%s: views %d and %d are the same (%d, %d)", who,
                   u, t, h_flip[t], h_shift[t]);
    v.flip[t] = h_flip[t];
    v.shift[t] = h_shift[t];
    v.c[t] = need_rotation ? h_cos[t] : 1.0;
    v.s[t] = need_rotation ? h_sin[t] : 0.0;
    PCLS_REQUIRE(isfinite(v.c[t]) && isfinite(v.s[t]), "%s: view %d: cos / sin not finite", who, t);
  }
  for (int t = n_views; t < TTA_MAX_VIEWS; ++t) { v.flip[t] = 0; v.shift[t] = 0; v.c[t] = 1.0; v.s[t] = 0.0; }
  return PCLS_OK;
}

static int tta_grid(int64_t blocks, int per_sm) {
  const int64_t cap = (int64_t)sm_count() * per_sm;
  return (int)std::max<int64_t>(1, std::min(blocks, cap));
}

}  // namespace pcls

using namespace pcls;

extern "C" int pcls_tta_views(const float* raw, int channels, int B, int H, int W, const double* h_mean5,
                              const double* h_std5, int n_views, const int* h_flip, const int* h_shift,
                              const double* h_cos, const double* h_sin, int precision, void* input8, uint8_t* mask,
                              pcls_stream stream) {
  PCLS_REQUIRE(B >= 0 && H > 0 && W > 0, "pcls_tta_views: bad sizes B=%d H=%d W=%d", B, H, W);
  PCLS_REQUIRE(channels == 5 || channels == 6, "pcls_tta_views: channels must be 5 or 6, got %d", channels);
  PCLS_REQUIRE(precision == PCLS_F16 || precision == PCLS_BF16, "pcls_tta_views: bad precision %d", precision);
  PCLS_REQUIRE(h_mean5 != nullptr && h_std5 != nullptr, "pcls_tta_views: h_mean5 / h_std5 must not be NULL");
  TtaViews v;
  int rc = tta_check_views("pcls_tta_views", W, n_views, h_flip, h_shift, h_cos, h_sin, true, v);
  if (rc) return rc;
  const int64_t n_pixels = (int64_t)B * H * W;
  PCLS_REQUIRE(n_pixels == 0 || (raw != nullptr && input8 != nullptr && mask != nullptr),
               "pcls_tta_views: raw / input8 / mask must not be NULL");
  if (n_pixels == 0) return PCLS_OK;
  TtaNorm nrm;
  for (int c = 0; c < 5; ++c) { nrm.mean[c] = h_mean5[c]; nrm.std[c] = h_std5[c]; }
  const int grid = tta_grid(ceil_div(n_pixels, 256), 16);
  if (precision == PCLS_F16)
    tta_views_kernel<__half><<<grid, 256, 0, (cudaStream_t)stream>>>(raw, channels, B, H, W, v, nrm, (int4*)input8, mask);
  else
    tta_views_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(raw, channels, B, H, W, v, nrm, (int4*)input8,
                                                                            mask);
  return check_launch("tta_views_kernel");
}

extern "C" int pcls_tta_merge(const float* probs, const uint8_t* mask, int B, int H, int W, int num_classes,
                              int none_index, int n_views, const int* h_flip, const int* h_shift, float* out_probs,
                              int32_t* out_preds, pcls_stream stream) {
  PCLS_REQUIRE(B >= 0 && H > 0 && W > 0, "pcls_tta_merge: bad sizes B=%d H=%d W=%d", B, H, W);
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= TTA_MAX_NC, "pcls_tta_merge: num_classes %d not in [1,%d]",
               num_classes, TTA_MAX_NC);
  PCLS_REQUIRE(none_index >= 0 && none_index < num_classes, "pcls_tta_merge: none_index %d not in [0,%d)", none_index,
               num_classes);
  TtaViews v;
  int rc = tta_check_views("pcls_tta_merge", W, n_views, h_flip, h_shift, nullptr, nullptr, false, v);
  if (rc) return rc;
  const int64_t n_pixels = (int64_t)B * H * W;
  PCLS_REQUIRE(n_pixels == 0 || (probs != nullptr && mask != nullptr && out_preds != nullptr),
               "pcls_tta_merge: probs / mask / out_preds must not be NULL");
  if (n_pixels == 0) return PCLS_OK;
  const int grid = tta_grid(ceil_div(ceil_div(n_pixels, 32), TTA_WARPS), 8);
  tta_merge_kernel<<<grid, TTA_WARPS * 32, 0, (cudaStream_t)stream>>>(probs, mask, B, H, W, num_classes, none_index, v,
                                                                       out_probs, out_preds);
  return check_launch("tta_merge_kernel");
}
