// Calibrated confidence (sm_100a): per-pixel confidence / entropy at a softmax temperature, the NLL of a grid of
// temperatures (the fit of post-hoc temperature scaling, Guo et al., ICML 2017), the reliability histogram that ECE / MCE
// come from, and the per-point confidence of the k-NN labels.  No reference call site: the reference reduces the softmax
// to an argmax.  The rules are stated in include/pclseg.h and restated in float64 by oracle/calibration.py.
//
// confidence_kernel: HBM-bound, NC*4 B read (+ NC*4 B probabilities written) + 1 B mask + 8 B conf / entropy written per
//   pixel.  Each warp stages 32 pixels x NC values through shared memory (coalesced, as head_kernel), lane = pixel.  In
//   logits mode v_c = z_c * a (rounded, __fmul_rn so that nvcc cannot fuse it into the softmax's subtraction) goes through
//   the head's own softmax_argmax: at a = 1 the probabilities are head_kernel's bits.
// temperature_nll_kernel: exp-bound (n_temps * NC expf per counted pixel).  A warp stages 32 pixels' logits; each lane
//   then owns one temperature (two above 32) and a subset of the 32 pixels (all of them at >= 32 temperatures; row reads
//   are shared-memory broadcasts), keeping its NLL sums in float64 registers for the whole grid-stride loop; per-block
//   float64 partials in shared memory, one global atomic per temperature per block.  max_c fl(z_c a) = fl(max_c z_c * a) for a > 0 (rounding is monotone), so the max is
//   taken once per pixel.
// reliability_kernel: 12 B read per element; per-block shared-memory histogram (int64 count / correct, float64 conf), one
//   global atomic per non-empty bin and block.
// point_confidence_kernel: one thread per point, 12 B read + a 4 B gather + 4 B written.
#include "nn_kernels.cuh"

#include <math.h>

namespace pcls {

constexpr int CAL_MAX_NC = 32;
constexpr int CAL_MAX_TEMPS = 64;
constexpr int CAL_MAX_BINS = 64;
constexpr int CAL_WARPS = 8;

struct CalTemps { float a[CAL_MAX_TEMPS]; };

__global__ void __launch_bounds__(CAL_WARPS * 32)
confidence_kernel(const float* __restrict__ src, bool is_logits, const uint8_t* __restrict__ mask, int64_t n, int nc,
                  float a, float* __restrict__ out_probs, float* __restrict__ out_conf, float* __restrict__ out_entropy) {
  __shared__ float tile[CAL_WARPS][32 * (CAL_MAX_NC + 1)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* t = tile[warp];
  const int pitch = nc + 1;
  const float log_nc = logf((float)nc);
  const int64_t n_groups = (n + 31) / 32;
  for (int64_t g = (int64_t)blockIdx.x * CAL_WARPS + warp; g < n_groups; g += (int64_t)gridDim.x * CAL_WARPS) {
    const int64_t p0 = g * 32;
    const int np = n - p0 >= 32 ? 32 : (int)(n - p0);
    const float* s = src + p0 * nc;
    const int n_el = np * nc;
    for (int e = lane; e < n_el; e += 32) t[(e / nc) * pitch + (e % nc)] = __ldg(s + e);
    __syncwarp();
    if (lane < np) {
      float v[CAL_MAX_NC];
#pragma unroll
      for (int c = 0; c < CAL_MAX_NC; ++c) v[c] = (c < nc) ? t[lane * pitch + c] : 0.0f;
      int best = 0;
      if (is_logits) {
#pragma unroll
        for (int c = 0; c < CAL_MAX_NC; ++c) if (c < nc) v[c] = __fmul_rn(v[c], a);
        best = softmax_argmax<CAL_MAX_NC>(v, nc);
      } else {
        float bp = -1.0f;
#pragma unroll
        for (int c = 0; c < CAL_MAX_NC; ++c) if (c < nc && v[c] > bp) { bp = v[c]; best = c; }
      }
      float top = 0.0f;
#pragma unroll
      for (int c = 0; c < CAL_MAX_NC; ++c) if (c == best) top = v[c];   // no dynamic index: v stays in registers
      const bool valid = mask == nullptr || mask[p0 + lane] != 0;
      if (out_conf != nullptr) out_conf[p0 + lane] = valid ? top : 0.0f;
      if (out_entropy != nullptr) out_entropy[p0 + lane] = valid ? normalised_entropy<CAL_MAX_NC>(v, nc, log_nc) : 0.0f;
      if (out_probs != nullptr && is_logits) {
#pragma unroll
        for (int c = 0; c < CAL_MAX_NC; ++c) if (c < nc) t[lane * pitch + c] = v[c];
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

__global__ void __launch_bounds__(CAL_WARPS * 32)
temperature_nll_kernel(const float* __restrict__ logits, const int32_t* __restrict__ label, int64_t n, int nc,
                       int ignore_index, int n_temps, CalTemps temps, double* __restrict__ nll_acc,
                       unsigned long long* __restrict__ counted) {
  __shared__ float tile[CAL_WARPS][32 * (CAL_MAX_NC + 1)];
  __shared__ int ylab[CAL_WARPS][32];
  __shared__ double part[CAL_MAX_TEMPS];
  __shared__ unsigned long long block_count;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < CAL_MAX_TEMPS; i += blockDim.x) part[i] = 0.0;
  if (threadIdx.x == 0) block_count = 0;
  __syncthreads();
  float* t = tile[warp];
  const int pitch = nc + 1;
  // lane -> (temperature, pixel subset): tp lanes (a power of two >= n_temps, at most 32) cover the temperatures, the
  // 32 / tp lane groups split the group's pixels; above 32 temperatures every lane owns two (lane and lane + 32)
  int tp = 1;
  while (tp < n_temps && tp < 32) tp <<= 1;
  const int n_sub = 32 / tp, t0 = lane % tp, t1 = t0 + 32;
  const bool two = n_temps > 32;
  unsigned sub_bits = 0;
  for (int j = lane / tp; j < 32; j += n_sub) sub_bits |= 1u << j;
  const float a0 = t0 < n_temps ? temps.a[t0] : 1.0f, a1 = t1 < n_temps ? temps.a[t1] : 1.0f;
  double acc0 = 0.0, acc1 = 0.0;
  unsigned int my_count = 0;
  const int64_t n_groups = (n + 31) / 32;
  for (int64_t g = (int64_t)blockIdx.x * CAL_WARPS + warp; g < n_groups; g += (int64_t)gridDim.x * CAL_WARPS) {
    const int64_t p0 = g * 32;
    const int np = n - p0 >= 32 ? 32 : (int)(n - p0);
    const int y_lane = lane < np ? __ldg(label + p0 + lane) : -1;
    const bool ok_lane = y_lane >= 0 && y_lane < nc && y_lane != ignore_index;
    const unsigned ok_mask = __ballot_sync(0xffffffffu, ok_lane);
    if (ok_mask == 0) continue;                               // warp-uniform: nothing counted in this group
    const float* s = logits + p0 * nc;
    const int n_el = np * nc;
    for (int e = lane; e < n_el; e += 32) t[(e / nc) * pitch + (e % nc)] = __ldg(s + e);
    ylab[warp][lane] = y_lane;
    __syncwarp();
    my_count += lane == 0 ? __popc(ok_mask) : 0;
    for (unsigned rest = ok_mask & sub_bits; rest != 0; rest &= rest - 1) {
      const int j = __ffs(rest) - 1;                          // this lane's counted pixels of the group, in order
      const int y = ylab[warp][j];
      float z[CAL_MAX_NC];
      float zmax = t[j * pitch];
#pragma unroll
      for (int c = 0; c < CAL_MAX_NC; ++c) {
        z[c] = c < nc ? t[j * pitch + c] : 0.0f;
        if (c < nc) zmax = fmaxf(zmax, z[c]);
      }
      const float zy = t[j * pitch + y];
      const float m0 = __fmul_rn(zmax, a0);
      float e0 = 0.0f;
      if (two) {
        const float m1 = __fmul_rn(zmax, a1);
        float e1 = 0.0f;
#pragma unroll
        for (int c = 0; c < CAL_MAX_NC; ++c) if (c < nc) {
          e0 = __fadd_rn(e0, expf(__fsub_rn(__fmul_rn(z[c], a0), m0)));
          e1 = __fadd_rn(e1, expf(__fsub_rn(__fmul_rn(z[c], a1), m1)));
        }
        acc1 += (double)__fsub_rn(__fadd_rn(logf(e1), m1), __fmul_rn(zy, a1));
      } else {
#pragma unroll
        for (int c = 0; c < CAL_MAX_NC; ++c) if (c < nc) e0 = __fadd_rn(e0, expf(__fsub_rn(__fmul_rn(z[c], a0), m0)));
      }
      acc0 += (double)__fsub_rn(__fadd_rn(logf(e0), m0), __fmul_rn(zy, a0));
    }
    __syncwarp();
  }
  if (t0 < n_temps) atomicAdd(part + t0, acc0);
  if (two && t1 < n_temps) atomicAdd(part + t1, acc1);
  if (my_count) atomicAdd(&block_count, (unsigned long long)my_count);
  __syncthreads();
  for (int i = threadIdx.x; i < n_temps; i += blockDim.x) atomicAdd(nll_acc + i, part[i]);
  if (threadIdx.x == 0 && block_count) atomicAdd(counted, block_count);
}

__global__ void __launch_bounds__(256)
reliability_kernel(const float* __restrict__ conf, const int32_t* __restrict__ pred, const int32_t* __restrict__ label,
                   int64_t n, int nc, int ignore_index, int n_bins, unsigned long long* __restrict__ bin_count,
                   unsigned long long* __restrict__ bin_correct, double* __restrict__ bin_conf) {
  __shared__ unsigned long long s_count[CAL_MAX_BINS], s_correct[CAL_MAX_BINS];
  __shared__ double s_conf[CAL_MAX_BINS];
  for (int i = threadIdx.x; i < n_bins; i += blockDim.x) { s_count[i] = 0; s_correct[i] = 0; s_conf[i] = 0.0; }
  __syncthreads();
  const float nb = (float)n_bins;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int y = __ldg(label + i), q = __ldg(pred + i);
    if (y < 0 || y >= nc || y == ignore_index || q < 0 || q >= nc) continue;
    const float c = __ldg(conf + i);
    const int b = max(0, min((int)__fmul_rn(c, nb), n_bins - 1));
    atomicAdd(s_count + b, 1ull);
    if (q == y) atomicAdd(s_correct + b, 1ull);
    atomicAdd(s_conf + b, (double)c);
  }
  __syncthreads();
  for (int b = threadIdx.x; b < n_bins; b += blockDim.x) {
    if (s_count[b] == 0) continue;
    atomicAdd(bin_count + b, s_count[b]);
    if (s_correct[b]) atomicAdd(bin_correct + b, s_correct[b]);
    atomicAdd(bin_conf + b, s_conf[b]);
  }
}

__device__ __forceinline__ int cal_scan_of(const int64_t* __restrict__ offsets, int B, int64_t i) {
  int lo = 0, hi = B;  // b with offsets[b] <= i < offsets[b+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(offsets + mid) <= i) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256)
point_confidence_kernel(const float* __restrict__ probs, const int64_t* __restrict__ offsets, int B, int H, int W,
                        int64_t total, const int32_t* __restrict__ proj_x, const int32_t* __restrict__ proj_y,
                        const int32_t* __restrict__ point_labels, int nc, float* __restrict__ out_conf) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int x = __ldg(proj_x + i), y = __ldg(proj_y + i), l = __ldg(point_labels + i);
    float c = 0.0f;
    if (x >= 0 && l >= 0 && l < nc) {
      const int b = cal_scan_of(offsets, B, i);
      c = __ldg(probs + (((int64_t)b * H + y) * W + x) * nc + l);
    }
    out_conf[i] = c;
  }
}

static int cal_grid(int64_t blocks, int per_sm) {
  const int64_t cap = (int64_t)sm_count() * per_sm;
  return (int)std::max<int64_t>(1, std::min(blocks, cap));
}

}  // namespace pcls

using namespace pcls;

extern "C" int pcls_confidence(const float* logits, const float* probs, const uint8_t* mask, int64_t n, int num_classes,
                               float inv_temperature, float* out_probs, float* out_conf, float* out_entropy,
                               pcls_stream stream) {
  PCLS_REQUIRE(n >= 0, "pcls_confidence: negative n");
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= CAL_MAX_NC, "pcls_confidence: num_classes %d not in [1,%d]",
               num_classes, CAL_MAX_NC);
  PCLS_REQUIRE((logits == nullptr) != (probs == nullptr), "pcls_confidence: exactly one of logits / probs must be given");
  PCLS_REQUIRE(isfinite(inv_temperature) && inv_temperature > 0.0f,
               "pcls_confidence: inv_temperature %g must be finite and > 0", (double)inv_temperature);
  PCLS_REQUIRE(logits != nullptr || inv_temperature == 1.0f,
               "pcls_confidence: probs mode needs inv_temperature 1, got %g", (double)inv_temperature);
  PCLS_REQUIRE(out_probs != nullptr || out_conf != nullptr || out_entropy != nullptr,
               "pcls_confidence: no output given (out_probs / out_conf / out_entropy are all NULL)");
  if (n == 0) return PCLS_OK;
  const bool is_logits = logits != nullptr;
  const int grid = cal_grid(ceil_div(ceil_div(n, 32), CAL_WARPS), 8);
  confidence_kernel<<<grid, CAL_WARPS * 32, 0, (cudaStream_t)stream>>>(is_logits ? logits : probs, is_logits, mask, n,
                                                                        num_classes, inv_temperature, out_probs,
                                                                        out_conf, out_entropy);
  return check_launch("confidence_kernel");
}

extern "C" int pcls_temperature_nll(const float* logits, const int32_t* label, int64_t n, int num_classes,
                                    int ignore_index, int n_temps, const float* h_inv_temps, double* nll_acc,
                                    int64_t* counted, pcls_stream stream) {
  PCLS_REQUIRE(n >= 0, "pcls_temperature_nll: negative n");
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= CAL_MAX_NC, "pcls_temperature_nll: num_classes %d not in [1,%d]",
               num_classes, CAL_MAX_NC);
  PCLS_REQUIRE(n_temps >= 1 && n_temps <= CAL_MAX_TEMPS, "pcls_temperature_nll: n_temps %d not in [1,%d]", n_temps,
               CAL_MAX_TEMPS);
  PCLS_REQUIRE(h_inv_temps != nullptr, "pcls_temperature_nll: h_inv_temps is NULL");
  CalTemps temps;
  for (int t = 0; t < CAL_MAX_TEMPS; ++t) {
    if (t < n_temps)
      PCLS_REQUIRE(isfinite(h_inv_temps[t]) && h_inv_temps[t] > 0.0f,
                   "pcls_temperature_nll: inverse temperature %d (%g) must be finite and > 0", t, (double)h_inv_temps[t]);
    temps.a[t] = t < n_temps ? h_inv_temps[t] : 1.0f;
  }
  PCLS_REQUIRE(n == 0 || (logits != nullptr && label != nullptr && nll_acc != nullptr && counted != nullptr),
               "pcls_temperature_nll: logits / label / nll_acc / counted must not be NULL");
  if (n == 0) return PCLS_OK;
  const int grid = cal_grid(ceil_div(ceil_div(n, 32), CAL_WARPS), 4);
  temperature_nll_kernel<<<grid, CAL_WARPS * 32, 0, (cudaStream_t)stream>>>(
      logits, label, n, num_classes, ignore_index, n_temps, temps, nll_acc, reinterpret_cast<unsigned long long*>(counted));
  return check_launch("temperature_nll_kernel");
}

extern "C" int pcls_reliability_update(const float* conf, const int32_t* pred, const int32_t* label, int64_t n,
                                       int num_classes, int ignore_index, int n_bins, int64_t* bin_count,
                                       int64_t* bin_correct, double* bin_conf, pcls_stream stream) {
  PCLS_REQUIRE(n >= 0, "pcls_reliability_update: negative n");
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= CAL_MAX_NC, "pcls_reliability_update: num_classes %d not in [1,%d]",
               num_classes, CAL_MAX_NC);
  PCLS_REQUIRE(n_bins >= 1 && n_bins <= CAL_MAX_BINS, "pcls_reliability_update: n_bins %d not in [1,%d]", n_bins,
               CAL_MAX_BINS);
  PCLS_REQUIRE(n == 0 || (conf != nullptr && pred != nullptr && label != nullptr && bin_count != nullptr &&
                          bin_correct != nullptr && bin_conf != nullptr),
               "pcls_reliability_update: conf / pred / label / bin_count / bin_correct / bin_conf must not be NULL");
  if (n == 0) return PCLS_OK;
  const int grid = cal_grid(ceil_div(n, 256 * 8), 8);
  reliability_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      conf, pred, label, n, num_classes, ignore_index, n_bins, reinterpret_cast<unsigned long long*>(bin_count),
      reinterpret_cast<unsigned long long*>(bin_correct), bin_conf);
  return check_launch("reliability_kernel");
}

extern "C" int pcls_point_confidence(const float* probs, const int64_t* offsets, int B, int H, int W, int64_t total,
                                     const int32_t* proj_x, const int32_t* proj_y, const int32_t* point_labels,
                                     int num_classes, float* out_conf, pcls_stream stream) {
  PCLS_REQUIRE(B >= 0 && H > 0 && W > 0 && total >= 0, "pcls_point_confidence: bad sizes B=%d H=%d W=%d total=%lld", B,
               H, W, (long long)total);
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= CAL_MAX_NC, "pcls_point_confidence: num_classes %d not in [1,%d]",
               num_classes, CAL_MAX_NC);
  PCLS_REQUIRE(total == 0 || B >= 1, "pcls_point_confidence: %lld points but no scan", (long long)total);
  PCLS_REQUIRE(total == 0 || (probs != nullptr && offsets != nullptr && proj_x != nullptr && proj_y != nullptr &&
                              point_labels != nullptr && out_conf != nullptr),
               "pcls_point_confidence: probs / offsets / proj_x / proj_y / point_labels / out_conf must not be NULL");
  if (total == 0) return PCLS_OK;
  const int grid = cal_grid(ceil_div(total, 256), 16);
  point_confidence_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(probs, offsets, B, H, W, total, proj_x, proj_y,
                                                                   point_labels, num_classes, out_conf);
  return check_launch("point_confidence_kernel");
}
