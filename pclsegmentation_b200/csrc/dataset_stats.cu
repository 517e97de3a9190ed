// Per-frame dataset statistics of range images (sm_100a): the moments behind a config's INPUT_MEAN / INPUT_STD, channel
// ranges, pixel occupancy per row / column and class counts.  Takes the place of the reference's offline numpy tool
// (preprocessing/inspect_training_data.py, SURVEY.md §2 row 16); the exact rules are this project's contract in
// include/pclseg.h, restated in numpy by oracle/dataset_stats.py.
//
// Layout: one 8-CTA cluster per frame, CTA k of the cluster owns rows [H*k/8, H*(k+1)/8).  A CTA walks its rows in chunks
// of 512 pixels: the chunk's bytes are read as a flat array of 16-byte vectors (the two partial vectors at its ends
// element by element, so no byte outside the frames is touched and no alignment beyond the element's is needed) into
// registers, stored to shared memory, and the next chunk's loads are issued before the current one is reduced.  A pixel
// is 20-48 bytes, so per-thread pixel loads would be strided; the flat copy keeps every warp load contiguous.
//
// Determinism: thread t always reduces pixels t and t + 256 of each chunk, the warp combines by a fixed xor-shuffle tree,
// the CTA its 8 warps in order, and CTA 0 of the cluster the 8 CTA partials in rank order, read from the other CTAs'
// shared memory.  The order depends on H, W and the channel count only - not on the batch size, the frame's position,
// the dtype or the SM count - so a frame's sums are the same bits in any batch.  The integer counters are summed with
// atomics (exact in any order): rows and classes once per CTA, columns once per frame (CTA k of the cluster adds column
// block k over all 8 CTAs).
//
// Measured (NVIDIA B200, 1000 W power limit, profiles/dataset_stats_bench_b200.json, 64 frames of 64x2048 resident in
// HBM): float64 x 6 channels 0.146 ms = 2.76 TB/s, 0.41 of the 6.65 TB/s HBM peak bench.py uses.  The kernel is not
// bandwidth-bound: float32 frames, half the bytes, take 0.131 ms.  The per-pixel work (conversion, 20 float64
// accumulations, the row / class warp matches, the column atomic) bounds it, at 118 registers = 2 CTAs per SM.
#include "common.cuh"

#include <atomic>
#include <cooperative_groups.h>
#include <math.h>

namespace cg = cooperative_groups;

namespace pcls {

constexpr int DS_THREADS = 256;
constexpr int DS_CHUNK_PX = 2 * DS_THREADS;   // pixels per staging step
constexpr int DS_CLUSTER = 8;                 // CTAs (row slices) per frame
constexpr int DS_MAX_NC = 32;
constexpr int DS_MAX_W = 16384;               // the column counters live in shared memory,
constexpr int DS_MAX_H = 16384;               // and the row counters of a CTA's H/8 rows
constexpr size_t DS_MAX_DYN = (DS_MAX_W + DS_MAX_H / DS_CLUSTER) * sizeof(unsigned);

struct Shift5 { double s[5]; };

template <typename T>
__device__ __forceinline__ void ds_load_vec(const char* lo, const char* hi, const char* a, uint4& r) {
  if (a >= lo && a + 16 <= hi) { r = __ldg(reinterpret_cast<const uint4*>(a)); return; }
  T e[16 / sizeof(T)];
#pragma unroll
  for (int j = 0; j < (int)(16 / sizeof(T)); ++j) {
    const char* p = a + j * sizeof(T);
    e[j] = (p >= lo && p < hi) ? __ldg(reinterpret_cast<const T*>(p)) : T(0);
  }
  memcpy(&r, e, 16);
}

template <typename T, int C>
__global__ void __cluster_dims__(DS_CLUSTER, 1, 1) __launch_bounds__(DS_THREADS)
dataset_stats_kernel(const T* __restrict__ frames, int H, int W, Shift5 sh, int nc, double* __restrict__ frame_sums,
                     int64_t* __restrict__ frame_valid, unsigned long long* __restrict__ row_valid,
                     unsigned long long* __restrict__ col_valid, unsigned long long* __restrict__ class_pixels,
                     unsigned long long* __restrict__ dropped) {
  constexpr int VEC = 16 / sizeof(T);                    // elements per 16-byte vector
  constexpr int NV = DS_CHUNK_PX * C / VEC + 1;          // vectors that cover a chunk at any 16-byte phase
  constexpr int VPT = (NV + DS_THREADS - 1) / DS_THREADS;
  __shared__ __align__(16) T stage[NV * VEC];
  __shared__ double part[20];                            // this CTA's (sum, sum sq, min, max) x 5 channels
  __shared__ double warp_part[DS_THREADS / 32][20];
  __shared__ unsigned long long part_valid;
  __shared__ unsigned warp_valid[DS_THREADS / 32];
  __shared__ unsigned cls_s[DS_MAX_NC + 1];              // [nc] = dropped
  extern __shared__ unsigned dyn_s[];                    // [W] column counters, then this CTA's row counters
  unsigned* col_s = dyn_s;
  unsigned* row_s = dyn_s + W;

  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int64_t f = blockIdx.x / DS_CLUSTER;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r0 = (int)((int64_t)H * rank / DS_CLUSTER), r1 = (int)((int64_t)H * (rank + 1) / DS_CLUSTER);
  for (int i = tid; i < W + (r1 - r0); i += DS_THREADS) dyn_s[i] = 0;
  if (tid <= DS_MAX_NC) cls_s[tid] = 0;

  double sum[5], sq[5], mn[5], mx[5];
#pragma unroll
  for (int c = 0; c < 5; ++c) { sum[c] = 0.0; sq[c] = 0.0; mn[c] = INFINITY; mx[c] = -INFINITY; }
  unsigned nvalid = 0;

  const char* fbase = reinterpret_cast<const char*>(frames + f * H * W * C);
  const int64_t p0 = (int64_t)r0 * W, p1 = (int64_t)r1 * W;
  uint4 reg[VPT];
  auto load_chunk = [&](int64_t q) {
    const int64_t n = p1 - q < DS_CHUNK_PX ? p1 - q : DS_CHUNK_PX;
    const char* lo = fbase + q * C * (int64_t)sizeof(T);
    const char* hi = lo + n * C * (int64_t)sizeof(T);
    const char* a0 = reinterpret_cast<const char*>(reinterpret_cast<uintptr_t>(lo) & ~(uintptr_t)15);
#pragma unroll
    for (int k = 0; k < VPT; ++k) {
      const int v = tid + k * DS_THREADS;
      const char* a = a0 + (int64_t)v * 16;
      if (v < NV && a < hi) ds_load_vec<T>(lo, hi, a, reg[k]);
    }
  };
  if (p0 < p1) load_chunk(p0);
  __syncthreads();                                        // counters zeroed

  for (int64_t q = p0; q < p1; q += DS_CHUNK_PX) {
    const int64_t n = p1 - q < DS_CHUNK_PX ? p1 - q : DS_CHUNK_PX;
    const int phase = (int)((reinterpret_cast<uintptr_t>(fbase + q * C * (int64_t)sizeof(T)) & 15) / sizeof(T));
#pragma unroll
    for (int k = 0; k < VPT; ++k) {
      const int v = tid + k * DS_THREADS;
      if (v < NV) reinterpret_cast<uint4*>(stage)[v] = reg[k];
    }
    __syncthreads();
    if (q + DS_CHUNK_PX < p1) load_chunk(q + DS_CHUNK_PX);  // in flight while this chunk is reduced
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int i = tid + j * DS_THREADS;
      const bool in = i < n;
      const T* px = stage + phase + i * C;
      double v[C];
#pragma unroll
      for (int c = 0; c < C; ++c) v[c] = in ? (double)px[c] : 0.0;
      const bool valid = in && v[4] > 0.0;                // NaN range: invalid
      if (valid) {
        ++nvalid;
#pragma unroll
        for (int c = 0; c < 5; ++c) {
          const double d = v[c] - sh.s[c];
          sum[c] += d;
          sq[c] = fma(d, d, sq[c]);
          mn[c] = v[c] < mn[c] ? v[c] : mn[c];            // a NaN value never replaces the running min / max
          mx[c] = v[c] > mx[c] ? v[c] : mx[c];
        }
      }
      const int64_t pix = q + i;
      const int row = in ? (int)(pix / W) : -1;
      if (valid) atomicAdd(col_s + (pix - (int64_t)row * W), 1u);
      // valid pixels per row: a warp's 32 pixels span at most a few rows, one shared atomic per row and warp
      const unsigned vb = __ballot_sync(0xffffffffu, valid);
      const unsigned peers = __match_any_sync(0xffffffffu, row);
      if (in && lane == __ffs(peers) - 1 && (vb & peers)) atomicAdd(row_s + (row - r0), (unsigned)__popc(vb & peers));
      if (C == 6) {
        int bin = -1;
        if (valid && nc > 0) {
          const double l = v[C - 1];
          const double t = trunc(l);                      // (int32_t) cast: toward zero
          bin = (isfinite(l) && t >= 0.0 && t < (double)nc) ? (int)t : nc;
        }
        const unsigned bp = __match_any_sync(0xffffffffu, bin);   // one shared atomic per class and warp
        if (bin >= 0 && lane == __ffs(bp) - 1) atomicAdd(cls_s + bin, (unsigned)__popc(bp));
      }
    }
    __syncthreads();                                      // stage free for the next chunk
  }

  // warp tree (fixed xor butterfly), then the 8 warps in order
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
#pragma unroll
    for (int c = 0; c < 5; ++c) {
      sum[c] += __shfl_xor_sync(0xffffffffu, sum[c], off);
      sq[c] += __shfl_xor_sync(0xffffffffu, sq[c], off);
      const double a = __shfl_xor_sync(0xffffffffu, mn[c], off), b = __shfl_xor_sync(0xffffffffu, mx[c], off);
      mn[c] = a < mn[c] ? a : mn[c];
      mx[c] = b > mx[c] ? b : mx[c];
    }
    nvalid += __shfl_xor_sync(0xffffffffu, nvalid, off);
  }
  if (lane == 0) {
#pragma unroll
    for (int c = 0; c < 5; ++c) {
      warp_part[warp][c * 4 + 0] = sum[c]; warp_part[warp][c * 4 + 1] = sq[c];
      warp_part[warp][c * 4 + 2] = mn[c]; warp_part[warp][c * 4 + 3] = mx[c];
    }
    warp_valid[warp] = nvalid;
  }
  __syncthreads();
  if (tid < 20) {
    const int k = tid & 3;
    double a = warp_part[0][tid];
    for (int w = 1; w < DS_THREADS / 32; ++w) {
      const double b = warp_part[w][tid];
      a = k < 2 ? a + b : (k == 2 ? (b < a ? b : a) : (b > a ? b : a));
    }
    part[tid] = a;
  }
  if (tid == 32) {
    unsigned long long s = 0;
    for (int w = 0; w < DS_THREADS / 32; ++w) s += warp_valid[w];
    part_valid = s;
  }
  __syncthreads();
  cluster.sync();                                         // every CTA's partials and counters are final

  if (rank == 0 && tid < 20) {                            // the 8 slices in rank order
    const int k = tid & 3;
    double a = part[tid];
    for (int r = 1; r < DS_CLUSTER; ++r) {
      const double b = cluster.map_shared_rank(part, r)[tid];
      a = k < 2 ? a + b : (k == 2 ? (b < a ? b : a) : (b > a ? b : a));
    }
    frame_sums[f * 20 + tid] = a;
  }
  if (rank == 0 && tid == 32) {
    unsigned long long s = 0;
    for (int r = 0; r < DS_CLUSTER; ++r) s += *cluster.map_shared_rank(&part_valid, r);
    frame_valid[f] = (int64_t)s;
  }
  if (col_valid != nullptr) {
    const int c0 = (int)((int64_t)W * rank / DS_CLUSTER), c1 = (int)((int64_t)W * (rank + 1) / DS_CLUSTER);
    for (int c = c0 + tid; c < c1; c += DS_THREADS) {
      unsigned long long s = 0;
      for (int r = 0; r < DS_CLUSTER; ++r) s += cluster.map_shared_rank(col_s, r)[c];
      if (s) atomicAdd(col_valid + c, s);
    }
  }
  if (row_valid != nullptr)
    for (int i = tid; i < r1 - r0; i += DS_THREADS)
      if (row_s[i]) atomicAdd(row_valid + r0 + i, (unsigned long long)row_s[i]);
  if (C == 6 && tid < nc && class_pixels != nullptr && cls_s[tid]) atomicAdd(class_pixels + tid, (unsigned long long)cls_s[tid]);
  if (C == 6 && tid == nc && dropped != nullptr && cls_s[nc]) atomicAdd(dropped, (unsigned long long)cls_s[nc]);
  cluster.sync();                                         // no CTA leaves while another reads its shared memory
}

template <typename T, int C>
static int launch_stats(const void* frames, int B, int H, int W, const Shift5& sh, int nc, double* frame_sums,
                        int64_t* frame_valid, int64_t* row_valid, int64_t* col_valid, int64_t* class_pixels,
                        int64_t* dropped, cudaStream_t s) {
  // the largest request the size checks admit, set once per device (the attribute bounds, it does not reserve)
  static std::atomic<uint64_t> attr_set{0};
  int dev = 0;
  PCLS_CHECK_CUDA(cudaGetDevice(&dev));
  const uint64_t bit = 1ull << (dev & 63);
  if (!(attr_set.load() & bit)) {
    PCLS_CHECK_CUDA(cudaFuncSetAttribute(dataset_stats_kernel<T, C>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)DS_MAX_DYN));
    attr_set.fetch_or(bit);
  }
  const size_t dyn = (size_t)(W + ceil_div(H, DS_CLUSTER)) * sizeof(unsigned);
  dataset_stats_kernel<T, C><<<(unsigned)B * DS_CLUSTER, DS_THREADS, dyn, s>>>(
      reinterpret_cast<const T*>(frames), H, W, sh, nc, frame_sums, frame_valid,
      reinterpret_cast<unsigned long long*>(row_valid), reinterpret_cast<unsigned long long*>(col_valid),
      reinterpret_cast<unsigned long long*>(class_pixels), reinterpret_cast<unsigned long long*>(dropped));
  return check_launch("dataset_stats_kernel");
}

}  // namespace pcls

using namespace pcls;

extern "C" int pcls_dataset_stats(const void* frames, int dtype, int channels, int B, int H, int W,
                                  const double* h_shift5, int num_classes, double* frame_sums, int64_t* frame_valid,
                                  int64_t* row_valid, int64_t* col_valid, int64_t* class_pixels, int64_t* dropped,
                                  pcls_stream stream) {
  PCLS_REQUIRE(dtype == 0 || dtype == 1, "pcls_dataset_stats: dtype %d is neither 0 (float32) nor 1 (float64)", dtype);
  PCLS_REQUIRE(channels == 5 || channels == 6, "pcls_dataset_stats: channels must be 5 or 6, got %d", channels);
  PCLS_REQUIRE(B >= 0 && B <= (1 << 26) && H > 0 && H <= DS_MAX_H && W > 0 && W <= DS_MAX_W,
               "pcls_dataset_stats: bad sizes B=%d H=%d W=%d (H <= %d, W <= %d)", B, H, W, DS_MAX_H, DS_MAX_W);
  PCLS_REQUIRE((class_pixels == nullptr && dropped == nullptr) ||
               (channels == 6 && num_classes >= 1 && num_classes <= DS_MAX_NC),
               "pcls_dataset_stats: class_pixels / dropped need 6 channels and 1 <= num_classes <= %d (got %d, %d)",
               DS_MAX_NC, channels, num_classes);
  Shift5 sh;
  for (int c = 0; c < 5; ++c) {
    sh.s[c] = h_shift5 ? h_shift5[c] : 0.0;
    PCLS_REQUIRE(isfinite(sh.s[c]), "pcls_dataset_stats: h_shift5[%d] is not finite", c);
  }
  if (B == 0) return PCLS_OK;
  PCLS_REQUIRE(frames != nullptr && frame_sums != nullptr && frame_valid != nullptr,
               "pcls_dataset_stats: frames / frame_sums / frame_valid must not be NULL");
  PCLS_REQUIRE((uintptr_t)frames % (dtype ? 8 : 4) == 0, "pcls_dataset_stats: frames are not aligned to their dtype");
  const int nc = (class_pixels != nullptr || dropped != nullptr) ? num_classes : 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype == 0)
    return channels == 5 ? launch_stats<float, 5>(frames, B, H, W, sh, nc, frame_sums, frame_valid, row_valid, col_valid, class_pixels, dropped, s)
                         : launch_stats<float, 6>(frames, B, H, W, sh, nc, frame_sums, frame_valid, row_valid, col_valid, class_pixels, dropped, s);
  return channels == 5 ? launch_stats<double, 5>(frames, B, H, W, sh, nc, frame_sums, frame_valid, row_valid, col_valid, class_pixels, dropped, s)
                       : launch_stats<double, 6>(frames, B, H, W, sh, nc, frame_sums, frame_valid, row_valid, col_valid, class_pixels, dropped, s);
}
