// Instance ids for thing-class points: connected components in the range image (sm_100a).  No reference call site: the
// reference reads instance ids from label files (SemLaserScan.set_label, inst = label >> 16) but never produces them.
// The rules are the contract in include/pclseg.h, restated in numpy by oracle/point_instances.py; bit parity with any
// published clustering code is not claimed.
//
// Six launches, all over caller-provided scratch ([B*H*W] 16-byte node words, then [B*H*W] i32 parent, [B*H*W] i32 size):
//   pixel pass    key -> winner -> label.  A node stores parent[p] = p and (x, y, z, bits(label)) as one 16-byte word,
//                 so that the neighbour reads of the union pass are coalesced; other pixels store parent[p] = -1.
//   union pass    one thread per node over the forward half of the window (every unordered pair once).  Lock-free
//                 union-find in the style of ECL-CC (Jaiganesh & Burtscher, HPDC 2018): find with path halving, the larger
//                 root hooked under the smaller with atomicCAS.  Parents only ever point to smaller pixel indices, so a
//                 root is its tree's minimum pixel index whatever order the hooks land in.
//   flatten pass  parent[p] = root for every node.
//   point pass    rule 4: the point's pixel's root, or -1; atomicAdd of 1 on the root's size; the root is stashed in
//                 `instances`.  Integer atomics: the sizes do not depend on their order.
//   number pass   one CTA per scan walks its H*W pixels in index order: a root whose size is >= min_points gets the next
//                 id (warp ballots, a scan over the warps' counts); size[root] is overwritten with the id (0 if too small).
//   final pass    instances[i] = id of the stashed root, 0 for -1.
// So the output is the same bits on every run.
#include "common.cuh"

#include <math.h>

namespace pcls {

constexpr int PI_MAX_RY = 4;
constexpr int PI_MAX_RX = 8;
constexpr int PI_NUMBER_THREADS = 1024;

struct InstanceScratch {
  float4* node;    // [n] (x, y, z, bits(label)) at nodes
  int* parent;     // [n] -1 = not a node
  int* size;       // [n] points per root, then the root's id
};

static inline int64_t pi_scratch_bytes(int64_t n) { return n * (int64_t)(sizeof(float4) + 2 * sizeof(int)); }

static inline InstanceScratch pi_carve(void* scratch, int64_t n) {
  InstanceScratch s;
  s.node = reinterpret_cast<float4*>(scratch);
  s.parent = reinterpret_cast<int*>(s.node + n);
  s.size = s.parent + n;
  return s;
}

// d^2 = (dx*dx + dy*dy) + dz*dz in float32 with separate roundings (no contraction into FMA)
__device__ __forceinline__ float dist2(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

__device__ __forceinline__ int scan_of_point(const int64_t* __restrict__ offsets, int B, int64_t i) {
  int lo = 0, hi = B;  // b with offsets[b] <= i < offsets[b+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(offsets + mid) <= i) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(256)
instances_pixel_kernel(const float* __restrict__ points, const unsigned long long* __restrict__ keys,
                       const int64_t* __restrict__ offsets, int n, int HW, const int32_t* __restrict__ labels,
                       unsigned thing_mask, InstanceScratch s) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t pp = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; pp < n; pp += stride) {
    const int p = (int)pp;
    const unsigned long long key = __ldg(keys + p);
    int parent = -1;
    if (key != ~0ull) {
      const int64_t i = __ldg(offsets + p / HW) + (int64_t)(key & 0xffffffffull);
      const int label = __ldg(labels + i);
      if ((unsigned)label < 32u && ((thing_mask >> label) & 1u)) {
        const float4 xyz = __ldg(reinterpret_cast<const float4*>(points) + i);
        s.node[p] = make_float4(xyz.x, xyz.y, xyz.z, __int_as_float(label));
        parent = p;
      }
    }
    s.parent[p] = parent;
    s.size[p] = 0;
  }
}

// Root of x.  Parent words change under our feet (other threads hook roots and halve paths), so every read goes
// through volatile: a cached stale parent could make find() return a node that is no longer a root.
__device__ __forceinline__ int find_root(volatile int* parent, int x) {
  int p = parent[x];
  while (p != x) {
    const int g = parent[p];
    if (g != p) parent[x] = g;   // path halving: g is an ancestor of x, and x is not a root (no CAS targets it)
    x = g;
    p = parent[x];
  }
  return x;
}

__device__ __forceinline__ void unite(int* parent, int a, int b) {
  volatile int* vp = parent;
  int ra = find_root(vp, a), rb = find_root(vp, b);
  while (ra != rb) {
    const int lo = ra < rb ? ra : rb, hi = ra < rb ? rb : ra;
    const int prev = atomicCAS(parent + hi, hi, lo);   // hook the larger root under the smaller
    if (prev == hi) return;
    ra = find_root(vp, prev);                        // hi was hooked meanwhile: continue from where it went
    rb = find_root(vp, lo);
  }
}

template <int RY, int RX>
__global__ void __launch_bounds__(256)
instances_union_kernel(int n, int H, int W, int wrap, float tau2, InstanceScratch s) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  if (s.parent[p] < 0) return;
  const int HW = H * W;
  const int base = p - p % HW;
  const int r = (p - base) / W, c = (p - base) - r * W;
  const float4 me = s.node[p];
#pragma unroll 1
  for (int dr = 0; dr <= RY; ++dr) {
    const int rr = r + dr;
    if (rr >= H) break;
    // the row's 2 RX + 1 window entries are tested first (independent loads, unrolled), then joined
    unsigned join = 0;
#pragma unroll
    for (int dc = -RX; dc <= RX; ++dc) {
      if (dr == 0 && dc <= 0) continue;             // forward half: each unordered pair once
      int cc = c + dc;
      if (cc < 0 || cc >= W) {
        if (!wrap) continue;
        cc = cc < 0 ? cc + W : cc - W;              // 2 rx < W: one wrap at most
      }
      const int q = base + rr * W + cc;
      if (s.parent[q] < 0) continue;                // not a node (parent words of nodes never become negative)
      const float4 o = s.node[q];
      if (__float_as_int(o.w) != __float_as_int(me.w)) continue;
      if (!(dist2(me.x, me.y, me.z, o.x, o.y, o.z) <= tau2)) continue;
      join |= 1u << (dc + RX);
    }
    while (join) {
      const int dc = __ffs(join) - 1 - RX;
      join &= join - 1;
      int cc = c + dc;
      cc = cc < 0 ? cc + W : (cc >= W ? cc - W : cc);
      unite(s.parent, p, base + rr * W + cc);
    }
  }
}

__global__ void __launch_bounds__(256) instances_flatten_kernel(int n, InstanceScratch s) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  int x = s.parent[p];
  if (x < 0 || x == p) return;
  int y = s.parent[x];
  while (y != x) { x = y; y = s.parent[x]; }        // no writer is left: plain reads
  s.parent[p] = x;
}

__global__ void __launch_bounds__(256)
instances_point_kernel(const float* __restrict__ points, const unsigned long long* __restrict__ keys,
                       const int64_t* __restrict__ offsets, int B, int H, int W, int64_t total,
                       const int32_t* __restrict__ proj_x, const int32_t* __restrict__ proj_y,
                       const int32_t* __restrict__ labels, float tau2, InstanceScratch s, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int px = __ldg(proj_x + i);
  int root = -1;
  if (px >= 0) {
    const int b = scan_of_point(offsets, B, i);
    const int p = (b * H + __ldg(proj_y + i)) * W + px;
    const int rp = s.parent[p];
    if (rp >= 0) {
      const int64_t win = __ldg(offsets + b) + (int64_t)(__ldg(keys + p) & 0xffffffffull);
      bool in = win == i;
      if (!in) {
        const float4 w = s.node[p];
        const float4 me = __ldg(reinterpret_cast<const float4*>(points) + i);
        in = __ldg(labels + i) == __float_as_int(w.w) && dist2(me.x, me.y, me.z, w.x, w.y, w.z) <= tau2;
      }
      if (in) {
        root = rp;
        atomicAdd(s.size + rp, 1);
      }
    }
  }
  out[i] = root;
}

// One CTA per scan: ids 1, 2, ... to the roots with size >= min_points, in increasing pixel index.  Warp w owns the
// w-th of 32 contiguous segments of the scan's pixels: pass 1 counts its ids (coalesced reads, ballots), a scan over the
// 32 warp counts gives each warp its first id, pass 2 hands them out in pixel order.
__device__ __forceinline__ bool keeps_id(const InstanceScratch& s, int p, int min_points) {
  return s.parent[p] == p && s.size[p] >= min_points;
}

__global__ void __launch_bounds__(PI_NUMBER_THREADS)
instances_number_kernel(int HW, int min_points, InstanceScratch s, int32_t* __restrict__ counts) {
  constexpr int NW = PI_NUMBER_THREADS / 32;
  __shared__ int warp_first[NW + 1];
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int seg = ((HW + NW - 1) / NW + 31) / 32 * 32;
  const int lo = warp * seg, hi = min(HW, lo + seg);
  const int base = b * HW;
  int n = 0;
#pragma unroll 4
  for (int t = lo + lane; t - lane < hi; t += 32)   // warp-uniform trip count: every lane takes part in the ballots
    n += __popc(__ballot_sync(0xffffffffu, t < hi && keeps_id(s, base + t, min_points)));
  if (lane == 0) warp_first[warp + 1] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    warp_first[0] = 0;
    for (int w = 1; w <= NW; ++w) warp_first[w] += warp_first[w - 1];
    counts[b] = warp_first[NW];
  }
  __syncthreads();
  int next = warp_first[warp] + 1;
  const unsigned below = (1u << lane) - 1u;
  for (int t = lo + lane; t - lane < hi; t += 32) {
    const int p = base + t;
    const bool root = t < hi && s.parent[p] == p;
    const bool keep = root && s.size[p] >= min_points;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (root) s.size[p] = keep ? next + __popc(bal & below) : 0;
    next += __popc(bal);
  }
}

__global__ void __launch_bounds__(256)
instances_final_kernel(int64_t total, const int* __restrict__ size, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int root = out[i];
  out[i] = root >= 0 ? size[root] : 0;
}

template <int RY, int RX>
static void launch_union(int n, int H, int W, int wrap, float tau2, const InstanceScratch& s, cudaStream_t st) {
  instances_union_kernel<RY, RX><<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(n, H, W, wrap, tau2, s);
}

template <int RY>
static void launch_union_rx(int rx, int n, int H, int W, int wrap, float tau2, const InstanceScratch& s,
                            cudaStream_t st) {
  switch (rx) {
    case 0: launch_union<RY, 0>(n, H, W, wrap, tau2, s, st); break;
    case 1: launch_union<RY, 1>(n, H, W, wrap, tau2, s, st); break;
    case 2: launch_union<RY, 2>(n, H, W, wrap, tau2, s, st); break;
    case 3: launch_union<RY, 3>(n, H, W, wrap, tau2, s, st); break;
    case 4: launch_union<RY, 4>(n, H, W, wrap, tau2, s, st); break;
    case 5: launch_union<RY, 5>(n, H, W, wrap, tau2, s, st); break;
    case 6: launch_union<RY, 6>(n, H, W, wrap, tau2, s, st); break;
    case 7: launch_union<RY, 7>(n, H, W, wrap, tau2, s, st); break;
    default: launch_union<RY, 8>(n, H, W, wrap, tau2, s, st); break;
  }
}

}  // namespace pcls

using namespace pcls;

extern "C" int64_t pcls_point_instances_scratch_bytes(int B, int H, int W) {
  PCLS_REQUIRE(B >= 0 && H > 0 && W > 0 && (int64_t)B * H * W < ((int64_t)1 << 31),
               "pcls_point_instances_scratch_bytes: bad sizes B=%d H=%d W=%d (B*H*W must be < 2^31)", B, H, W);
  return pi_scratch_bytes((int64_t)B * H * W);
}

extern "C" int pcls_point_instances(const float* points, const uint64_t* keys, const int64_t* offsets, int B, int H,
                                    int W, int64_t total_points, const int32_t* proj_x, const int32_t* proj_y,
                                    const int32_t* point_labels, int num_classes, uint32_t thing_mask, int ry, int rx,
                                    int wrap, float tau, int min_points, void* scratch, int32_t* instances,
                                    int32_t* instance_counts, pcls_stream stream) {
  PCLS_REQUIRE(B >= 0 && H > 0 && W > 0 && total_points >= 0,
               "pcls_point_instances: bad sizes B=%d H=%d W=%d total=%lld", B, H, W, (long long)total_points);
  PCLS_REQUIRE((int64_t)B * H * W < ((int64_t)1 << 31), "pcls_point_instances: B*H*W = %lld must be < 2^31",
               (long long)B * H * W);
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= 32, "pcls_point_instances: num_classes %d not in [1,32]",
               num_classes);
  PCLS_REQUIRE(num_classes == 32 || (thing_mask >> num_classes) == 0,
               "pcls_point_instances: thing_mask 0x%x names a class >= num_classes %d", thing_mask, num_classes);
  PCLS_REQUIRE(ry >= 0 && ry <= PI_MAX_RY, "pcls_point_instances: ry %d not in [0,%d]", ry, PI_MAX_RY);
  PCLS_REQUIRE(rx >= 0 && rx <= PI_MAX_RX, "pcls_point_instances: rx %d not in [0,%d]", rx, PI_MAX_RX);
  PCLS_REQUIRE(ry + rx > 0, "pcls_point_instances: ry + rx must be > 0 (the window has no neighbour)");
  PCLS_REQUIRE(wrap == 0 || wrap == 1, "pcls_point_instances: wrap %d must be 0 or 1", wrap);
  PCLS_REQUIRE(!wrap || 2 * rx < W, "pcls_point_instances: wrap needs 2 rx < W (rx %d, W %d)", rx, W);
  PCLS_REQUIRE(isfinite(tau) && tau > 0.0f, "pcls_point_instances: tau %g must be finite and > 0", (double)tau);
  PCLS_REQUIRE(min_points >= 1, "pcls_point_instances: min_points %d must be >= 1", min_points);
  PCLS_REQUIRE(offsets != nullptr, "pcls_point_instances: offsets is NULL");
  if (B == 0) return PCLS_OK;
  PCLS_REQUIRE(keys != nullptr && scratch != nullptr && instance_counts != nullptr,
               "pcls_point_instances: keys / scratch / instance_counts must not be NULL");
  PCLS_REQUIRE(reinterpret_cast<uintptr_t>(scratch) % 16 == 0, "pcls_point_instances: scratch must be 16-byte aligned");
  PCLS_REQUIRE(total_points == 0 || (points != nullptr && proj_x != nullptr && proj_y != nullptr &&
                                     point_labels != nullptr && instances != nullptr),
               "pcls_point_instances: points / proj_x / proj_y / point_labels / instances must not be NULL");
  PCLS_REQUIRE(total_points == 0 || reinterpret_cast<uintptr_t>(points) % 16 == 0,
               "pcls_point_instances: points must be 16-byte aligned");
  const float tau2 = tau * tau;
  const int n = B * H * W;
  const InstanceScratch s = pi_carve(scratch, n);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t pblocks = ceil_div(n, 256), cap = (int64_t)sm_count() * 16;
  instances_pixel_kernel<<<(unsigned)(pblocks < cap ? pblocks : cap), 256, 0, st>>>(
      points, reinterpret_cast<const unsigned long long*>(keys), offsets, n, H * W, point_labels, thing_mask, s);
  int rc = check_launch("instances_pixel_kernel");
  if (rc != PCLS_OK) return rc;
  switch (ry) {
    case 0: launch_union_rx<0>(rx, n, H, W, wrap, tau2, s, st); break;
    case 1: launch_union_rx<1>(rx, n, H, W, wrap, tau2, s, st); break;
    case 2: launch_union_rx<2>(rx, n, H, W, wrap, tau2, s, st); break;
    case 3: launch_union_rx<3>(rx, n, H, W, wrap, tau2, s, st); break;
    default: launch_union_rx<4>(rx, n, H, W, wrap, tau2, s, st); break;
  }
  if ((rc = check_launch("instances_union_kernel")) != PCLS_OK) return rc;
  instances_flatten_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(n, s);
  if ((rc = check_launch("instances_flatten_kernel")) != PCLS_OK) return rc;
  if (total_points > 0) {
    instances_point_kernel<<<(unsigned)ceil_div(total_points, 256), 256, 0, st>>>(
        points, reinterpret_cast<const unsigned long long*>(keys), offsets, B, H, W, total_points, proj_x, proj_y,
        point_labels, tau2, s, instances);
    if ((rc = check_launch("instances_point_kernel")) != PCLS_OK) return rc;
  }
  instances_number_kernel<<<(unsigned)B, PI_NUMBER_THREADS, 0, st>>>(H * W, min_points, s, instance_counts);
  if ((rc = check_launch("instances_number_kernel")) != PCLS_OK) return rc;
  if (total_points > 0) {
    instances_final_kernel<<<(unsigned)ceil_div(total_points, 256), 256, 0, st>>>(total_points, s.size, instances);
    if ((rc = check_launch("instances_final_kernel")) != PCLS_OK) return rc;
  }
  return PCLS_OK;
}
