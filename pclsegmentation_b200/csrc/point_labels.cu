// Per-point labels from the range-image predictions (sm_100a).  No reference call site: the reference stops at the
// [H,W] predictions (inference.py:78).  The k-NN vote follows the post-processing published with RangeNet++ (Milioto et
// al., IROS 2019); the exact rules are the contract in include/pclseg.h, restated in numpy by oracle/point_labels.py.
//
// search == 1: each point takes its own pixel's prediction - one gather per point.
// search >  1: two passes.
//   pixel pass  one word per pixel: (bits of the winner's range) << 32 | prediction, ~0 for an empty pixel.  The winner's
//               range is read through the key's low word (its local index) from unproj_range, for both projection
//               variants (ring keys carry ~index, not the depth, in the high word).  24 B per pixel.
//   point pass  one thread per point: px / py / range read coalesced, the search^2 window words through L1.  Candidates
//               are packed as (bits(d) << 32 | j << 8 | label): d >= 0, so the integer order of the keys is "smaller d,
//               then lower j", the selection's tie rule.  The k smallest stay sorted in registers; the vote over them
//               runs in registers too.  16 B per point.
//               Measured on scans whose points come in random order (DESIGN.md §3): the point pass runs at 0.04-0.06 of
//               the HBM peak on these bytes - its cost is the window gathers, which neighbouring threads do not share.
//
// Bit-exactness: d = |rho_j - rho| * w_j is spelled with _rn intrinsics so that numpy float32 reproduces it.
#include "common.cuh"

#include <math.h>

namespace pcls {

constexpr int PL_MAX_SEARCH = 9;
constexpr int PL_MAX_K = 32;
constexpr int PL_MAX_NC = 32;
constexpr int PL_SMALL_K = 8;

struct WindowWeights { float w[PL_MAX_SEARCH * PL_MAX_SEARCH]; };

__device__ __forceinline__ int scan_of(const int64_t* __restrict__ offsets, int B, int64_t i) {
  int lo = 0, hi = B;  // b with offsets[b] <= i < offsets[b+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(offsets + mid) <= i) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256)
point_labels_direct_kernel(const int32_t* __restrict__ preds, const int64_t* __restrict__ offsets, int B, int H, int W,
                           int64_t total, const int32_t* __restrict__ proj_x, const int32_t* __restrict__ proj_y,
                           int none_index, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int px = __ldg(proj_x + i);
  int label = none_index;
  if (px >= 0) {
    const int b = scan_of(offsets, B, i);
    label = __ldg(preds + ((int64_t)b * H + __ldg(proj_y + i)) * W + px);
  }
  out[i] = label;
}

__global__ void __launch_bounds__(256)
point_labels_pixel_kernel(const int32_t* __restrict__ preds, const unsigned long long* __restrict__ keys,
                          const int64_t* __restrict__ offsets, int64_t n_pixels, int HW,
                          const float* __restrict__ unproj_range, unsigned long long* __restrict__ scratch) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t pix = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pix < n_pixels; pix += stride) {
    const unsigned long long key = __ldg(keys + pix);
    unsigned long long word = ~0ull;
    if (key != ~0ull) {
      const float rho = __ldg(unproj_range + __ldg(offsets + pix / HW) + (int64_t)(key & 0xffffffffull));
      word = ((unsigned long long)__float_as_uint(rho) << 32) | (unsigned long long)(uint32_t)__ldg(preds + pix);
    }
    scratch[pix] = word;
  }
}

// KL = capacity of the register list of selected entries (>= k): min(S*S, 32) in general, PL_SMALL_K when k is at most
// that (S >= 5) - the defaults (S 5, k 5) then keep 8 instead of 25 64-bit keys live: 48 instead of 110 registers.
template <int S, int KL>
__global__ void __launch_bounds__(256)
point_labels_knn_kernel(const unsigned long long* __restrict__ scratch, const int64_t* __restrict__ offsets, int B,
                        int H, int W, int64_t total, const int32_t* __restrict__ proj_x,
                        const int32_t* __restrict__ proj_y, const float* __restrict__ unproj_range, int none_index,
                        int k, WindowWeights wt, float cutoff, int ignore_class, int32_t* __restrict__ out) {
  constexpr int P = (S - 1) / 2;
  constexpr int KMAX = KL;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int px = __ldg(proj_x + i);
  if (px < 0) { out[i] = none_index; return; }
  const int py = __ldg(proj_y + i);
  const float rho = __ldg(unproj_range + i);
  const int b = scan_of(offsets, B, i);
  const unsigned long long* img = scratch + (int64_t)b * H * W;

  unsigned long long best[KMAX];  // the k smallest candidate keys, ascending; ~0 = unused
#pragma unroll
  for (int t = 0; t < KMAX; ++t) best[t] = ~0ull;
  int centre_label = 0;
#pragma unroll
  for (int dy = -P; dy <= P; ++dy) {
    const int r = py + dy;
#pragma unroll
    for (int dx = -P; dx <= P; ++dx) {
      const int c = px + dx;
      const int j = (dy + P) * S + (dx + P);
      if (r < 0 || r >= H || c < 0 || c >= W) continue;   // outside the image: invalid, no wrap-around
      const unsigned long long word = __ldg(img + (int64_t)r * W + c);
      if (word == ~0ull) continue;                          // empty pixel
      const int label = (int)(uint32_t)word;
      const float rho_j = (dy == 0 && dx == 0) ? rho : __uint_as_float((uint32_t)(word >> 32));
      if (dy == 0 && dx == 0) centre_label = label;
      const float d = __fmul_rn(fabsf(__fsub_rn(rho_j, rho)), wt.w[j]);
      unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | ((unsigned)j << 8) | (unsigned)(label & 0xff);
      // insertion into the sorted list: only its first k entries matter
#pragma unroll
      for (int t = 0; t < KMAX; ++t) {
        if (t >= k) break;
        const unsigned long long lo = key < best[t] ? key : best[t];
        key = key < best[t] ? best[t] : key;
        best[t] = lo;
      }
    }
  }
  // vote: the class with most votes, ties to the lowest class; score = count << 8 | (255 - label)
  unsigned best_score = 0;
#pragma unroll
  for (int t = 0; t < KMAX; ++t) {
    if (t >= k) break;
    const unsigned long long a = best[t];
    const bool va = a != ~0ull && (cutoff <= 0.0f || __uint_as_float((uint32_t)(a >> 32)) <= cutoff) &&
                    (int)(a & 0xff) != ignore_class;
    if (!va) continue;
    unsigned cnt = 0;
#pragma unroll
    for (int u = 0; u < KMAX; ++u) {
      if (u >= k) break;
      const unsigned long long e = best[u];
      const bool ve = e != ~0ull && (cutoff <= 0.0f || __uint_as_float((uint32_t)(e >> 32)) <= cutoff);
      cnt += (ve && (e & 0xff) == (a & 0xff)) ? 1u : 0u;
    }
    const unsigned score = (cnt << 8) | (255u - (unsigned)(a & 0xff));
    best_score = score > best_score ? score : best_score;
  }
  out[i] = best_score ? (int)(255u - (best_score & 0xff)) : centre_label;
}

__global__ void __launch_bounds__(256)
map_labels_kernel(const uint32_t* __restrict__ labels, int64_t n, const int32_t* __restrict__ lut, int lut_len,
                  int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int sem = (int)(__ldg(labels + i) & 0xFFFFu);
  out[i] = lut ? (sem < lut_len ? __ldg(lut + sem) : 0) : sem;
}

template <int S>
static void launch_knn(int64_t total, cudaStream_t s, const unsigned long long* scratch, const int64_t* offsets, int B,
                       int H, int W, const int32_t* proj_x, const int32_t* proj_y, const float* unproj_range,
                       int none_index, int k, const WindowWeights& wt, float cutoff, int ignore_class, int32_t* out) {
  constexpr int KFULL = S * S < PL_MAX_K ? S * S : PL_MAX_K;
  constexpr int KSMALL = S > 3 ? PL_SMALL_K : KFULL;   // S 3: the full list is 9 entries already
  const unsigned grid = (unsigned)ceil_div(total, 256);
  if (k <= KSMALL)
    point_labels_knn_kernel<S, KSMALL><<<grid, 256, 0, s>>>(
        scratch, offsets, B, H, W, total, proj_x, proj_y, unproj_range, none_index, k, wt, cutoff, ignore_class, out);
  else
    point_labels_knn_kernel<S, KFULL><<<grid, 256, 0, s>>>(
        scratch, offsets, B, H, W, total, proj_x, proj_y, unproj_range, none_index, k, wt, cutoff, ignore_class, out);
}

}  // namespace pcls

using namespace pcls;

extern "C" int pcls_point_labels(const int32_t* preds, const uint64_t* keys, const int64_t* offsets, int B, int H, int W,
                                 int64_t total_points, const int32_t* proj_x, const int32_t* proj_y,
                                 const float* unproj_range, int num_classes, int none_index, int search, int k,
                                 const float* h_window_weights, float cutoff, int ignore_class, uint64_t* pixel_scratch,
                                 int32_t* point_labels, pcls_stream stream) {
  PCLS_REQUIRE(B >= 0 && H > 0 && W > 0 && total_points >= 0, "pcls_point_labels: bad sizes B=%d H=%d W=%d total=%lld",
               B, H, W, (long long)total_points);
  PCLS_REQUIRE(search >= 1 && search <= PL_MAX_SEARCH && search % 2 == 1,
               "pcls_point_labels: search %d must be odd and in [1,%d]", search, PL_MAX_SEARCH);
  const int kmax = search * search < PL_MAX_K ? search * search : PL_MAX_K;
  PCLS_REQUIRE(k >= 1 && k <= kmax, "pcls_point_labels: k %d not in [1,%d] (search %d)", k, kmax, search);
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= PL_MAX_NC, "pcls_point_labels: num_classes %d not in [1,%d]",
               num_classes, PL_MAX_NC);
  PCLS_REQUIRE(none_index >= 0 && none_index < num_classes, "pcls_point_labels: none_index %d not in [0,%d)", none_index,
               num_classes);
  PCLS_REQUIRE(ignore_class == -1 || (ignore_class >= 0 && ignore_class < num_classes),
               "pcls_point_labels: ignore_class %d is neither -1 nor in [0,%d)", ignore_class, num_classes);
  PCLS_REQUIRE(search == 1 || pixel_scratch != nullptr, "pcls_point_labels: pixel_scratch is NULL with search %d > 1",
               search);
  PCLS_REQUIRE(!(cutoff != cutoff), "pcls_point_labels: cutoff is NaN");
  WindowWeights wt;
  for (int j = 0; j < search * search; ++j) {
    const float w = h_window_weights ? h_window_weights[j] : 1.0f;
    PCLS_REQUIRE(isfinite(w) && w >= 0.0f, "pcls_point_labels: h_window_weights[%d] = %g must be finite and >= 0", j,
                 (double)w);
    wt.w[j] = w + 0.0f;  // -0 -> +0: every distance is then a non-negative float whose bits order like its value
  }
  PCLS_REQUIRE(offsets != nullptr, "pcls_point_labels: offsets is NULL");
  if (total_points == 0 || B == 0) return PCLS_OK;
  PCLS_REQUIRE(preds != nullptr && proj_x != nullptr && proj_y != nullptr && point_labels != nullptr,
               "pcls_point_labels: preds / proj_x / proj_y / point_labels must not be NULL");
  PCLS_REQUIRE(search == 1 || (keys != nullptr && unproj_range != nullptr),
               "pcls_point_labels: keys / unproj_range must not be NULL with search > 1");
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned grid = (unsigned)ceil_div(total_points, 256);
  if (search == 1) {
    point_labels_direct_kernel<<<grid, 256, 0, s>>>(preds, offsets, B, H, W, total_points, proj_x, proj_y, none_index,
                                                    point_labels);
    return check_launch("point_labels_direct_kernel");
  }
  const int64_t n_pixels = (int64_t)B * H * W;
  int64_t pblocks = ceil_div(n_pixels, 256), cap = (int64_t)sm_count() * 16;
  point_labels_pixel_kernel<<<(unsigned)(pblocks < cap ? pblocks : cap), 256, 0, s>>>(
      preds, reinterpret_cast<const unsigned long long*>(keys), offsets, n_pixels, H * W, unproj_range,
      reinterpret_cast<unsigned long long*>(pixel_scratch));
  int rc = check_launch("point_labels_pixel_kernel");
  if (rc != PCLS_OK) return rc;
  const unsigned long long* sc = reinterpret_cast<const unsigned long long*>(pixel_scratch);
  switch (search) {
    case 3: launch_knn<3>(total_points, s, sc, offsets, B, H, W, proj_x, proj_y, unproj_range, none_index, k, wt, cutoff, ignore_class, point_labels); break;
    case 5: launch_knn<5>(total_points, s, sc, offsets, B, H, W, proj_x, proj_y, unproj_range, none_index, k, wt, cutoff, ignore_class, point_labels); break;
    case 7: launch_knn<7>(total_points, s, sc, offsets, B, H, W, proj_x, proj_y, unproj_range, none_index, k, wt, cutoff, ignore_class, point_labels); break;
    default: launch_knn<9>(total_points, s, sc, offsets, B, H, W, proj_x, proj_y, unproj_range, none_index, k, wt, cutoff, ignore_class, point_labels); break;
  }
  return check_launch("point_labels_knn_kernel");
}

extern "C" int pcls_map_labels(const uint32_t* labels, int64_t n, const int32_t* label_lut, int lut_len, int32_t* out,
                               pcls_stream stream) {
  PCLS_REQUIRE(n >= 0, "pcls_map_labels: n %lld < 0", (long long)n);
  PCLS_REQUIRE(label_lut == nullptr || lut_len >= 0, "pcls_map_labels: lut_len %d < 0", lut_len);
  if (n == 0) return PCLS_OK;
  PCLS_REQUIRE(labels != nullptr && out != nullptr, "pcls_map_labels: labels / out must not be NULL");
  map_labels_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(labels, n, label_lut, lut_len, out);
  return check_launch("map_labels_kernel");
}
