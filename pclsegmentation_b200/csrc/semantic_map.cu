// Semantic map fusion (sm_100a): the point labels of a pose-registered sequence voted into a voxel hash map, and points
// relabelled from it.  No reference call site.  The rules are the contract in include/pclseg.h, restated in numpy by
// oracle/semantic_map.py; parity with any published mapping code is not claimed.
//
// The table is open addressing with linear probing over `capacity` (a power of two) u64 keys, ~0 = empty, and a row of
// NC u32 vote counts per slot.  A key is claimed with a 64-bit atomicCAS and never released, so a slot seen holding a
// key holds it for good: a plain read that sees a key is exact, a stale "empty" read only costs a failed CAS.  Counts
// are integer atomics, so the set of (key, counts) does not depend on the order the atomics land in; only the slot a key
// takes does, and nothing observable depends on that.
//
// The world coordinates compile to DMUL / DADD only.  The DFMAs in the SASS are the division's own reciprocal and
// correction steps, which give the correctly rounded quotient (the IEEE division numpy performs).
//
// Launches: vote (one thread per point), grow (two memsets for the new table, then one thread per old slot), query (one
// thread per point).
#include "common.cuh"

#include <math.h>

namespace pcls {

constexpr int64_t SM_HALF = (int64_t)1 << 20;   // voxel indices in [-2^20, 2^20)
constexpr unsigned long long SM_EMPTY = ~0ull;

__device__ __forceinline__ int sm_scan_of_point(const int64_t* __restrict__ offsets, int B, int64_t i) {
  int lo = 0, hi = B;  // b with offsets[b] <= i < offsets[b+1]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(offsets + mid) <= i) lo = mid; else hi = mid;
  }
  return lo;
}

// w = ((r0*x + r1*y) + r2*z) + t in float64 with every product and sum rounded on its own: no DFMA, so the numpy oracle
// computes the same bits.
__device__ __forceinline__ double world(const double* __restrict__ row, double x, double y, double z) {
  return __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(__ldg(row), x), __dmul_rn(__ldg(row + 1), y)),
                             __dmul_rn(__ldg(row + 2), z)), __ldg(row + 3));
}

__device__ __forceinline__ bool voxel_index(double w, double s, int64_t* v) {
  if (!isfinite(w)) return false;
  const double f = floor(__ddiv_rn(w, s));
  if (!(f >= -(double)SM_HALF && f < (double)SM_HALF)) return false;
  *v = (int64_t)f + SM_HALF;
  return true;
}

// The key of a point of scan b, or false when it has no voxel.
__device__ __forceinline__ bool voxel_key(const double* __restrict__ pose, float x, float y, float z, double s,
                                          unsigned long long* key) {
  const double dx = x, dy = y, dz = z;
  int64_t vx, vy, vz;
  if (!voxel_index(world(pose, dx, dy, dz), s, &vx)) return false;
  if (!voxel_index(world(pose + 4, dx, dy, dz), s, &vy)) return false;
  if (!voxel_index(world(pose + 8, dx, dy, dz), s, &vz)) return false;
  *key = ((unsigned long long)vx << 42) | ((unsigned long long)vy << 21) | (unsigned long long)vz;
  return true;
}

__device__ __forceinline__ unsigned long long sm_hash(unsigned long long k) {   // MurmurHash3's 64-bit finaliser
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ull;
  k ^= k >> 33;
  return k;
}

// Slot of `key`, inserting it if new (state[0] += 1 on the claiming CAS); -1 after `capacity` probes without a free slot.
__device__ __forceinline__ int64_t insert_key(unsigned long long* keys, int64_t capacity, unsigned long long key,
                                              int64_t* state) {
  const unsigned long long mask = (unsigned long long)capacity - 1;
  unsigned long long slot = sm_hash(key) & mask;
  for (int64_t p = 0; p < capacity; ++p, slot = (slot + 1) & mask) {
    unsigned long long k = __ldcg(keys + slot);
    if (k == SM_EMPTY) {
      k = atomicCAS(keys + slot, SM_EMPTY, key);
      if (k == SM_EMPTY) {
        atomicAdd(reinterpret_cast<unsigned long long*>(state), 1ull);
        return (int64_t)slot;
      }
    }
    if (k == key) return (int64_t)slot;
  }
  return -1;
}

__global__ void __launch_bounds__(256)
map_vote_kernel(const float* __restrict__ points, const int64_t* __restrict__ offsets, int B, int64_t total,
                const double* __restrict__ poses, double s, double min2, double max2, const int32_t* __restrict__ labels,
                int nc, int ignore_class, unsigned long long* keys, unsigned* counts, int64_t capacity,
                int64_t* state) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int label = __ldg(labels + i);
  if (label < 0 || label >= nc || label == ignore_class) return;
  const float4 p = __ldg(reinterpret_cast<const float4*>(points) + i);
  const double x = p.x, y = p.y, z = p.z;
  const double r2 = __dadd_rn(__dadd_rn(__dmul_rn(x, x), __dmul_rn(y, y)), __dmul_rn(z, z));
  if (!(r2 >= min2) || (max2 > 0.0 && !(r2 <= max2))) return;
  unsigned long long key;
  if (!voxel_key(poses + 12 * sm_scan_of_point(offsets, B, i), p.x, p.y, p.z, s, &key)) return;
  const int64_t slot = insert_key(keys, capacity, key, state);
  if (slot < 0) {
    atomicAdd(reinterpret_cast<unsigned long long*>(state + 1), 1ull);
    return;
  }
  atomicAdd(counts + slot * nc + label, 1u);
}

__global__ void __launch_bounds__(256)
map_grow_kernel(const unsigned long long* __restrict__ old_keys, const unsigned* __restrict__ old_counts,
                int64_t old_capacity, int nc, unsigned long long* new_keys, unsigned* __restrict__ new_counts,
                int64_t new_capacity, int64_t* state) {
  const int64_t o = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= old_capacity) return;
  const unsigned long long key = __ldg(old_keys + o);
  if (key == SM_EMPTY) return;
  // every key is distinct, so each CAS claims a fresh slot; the occupied count is unchanged
  const unsigned long long mask = (unsigned long long)new_capacity - 1;
  unsigned long long slot = sm_hash(key) & mask;
  int64_t p = 0;
  for (; p < new_capacity; ++p, slot = (slot + 1) & mask)
    if (atomicCAS(new_keys + slot, SM_EMPTY, key) == SM_EMPTY) break;
  if (p == new_capacity) {
    atomicAdd(reinterpret_cast<unsigned long long*>(state + 1), 1ull);
    return;
  }
  for (int c = 0; c < nc; ++c) new_counts[slot * nc + c] = __ldg(old_counts + o * nc + c);
}

__global__ void __launch_bounds__(256)
map_query_kernel(const float* __restrict__ points, const int64_t* __restrict__ offsets, int B, int64_t total,
                 const double* __restrict__ poses, double s, const int32_t* __restrict__ labels_in, int nc,
                 unsigned keep_mask, int min_votes, const unsigned long long* __restrict__ keys,
                 const unsigned* __restrict__ counts, int64_t capacity, int32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int label = __ldg(labels_in + i);
  out[i] = label;
  if ((unsigned)label < 32u && ((keep_mask >> label) & 1u)) return;
  const float4 p = __ldg(reinterpret_cast<const float4*>(points) + i);
  unsigned long long key;
  if (!voxel_key(poses + 12 * sm_scan_of_point(offsets, B, i), p.x, p.y, p.z, s, &key)) return;
  const unsigned long long mask = (unsigned long long)capacity - 1;
  unsigned long long slot = sm_hash(key) & mask;
  for (int64_t q = 0; q < capacity; ++q, slot = (slot + 1) & mask) {
    const unsigned long long k = __ldg(keys + slot);
    if (k == SM_EMPTY) return;
    if (k != key) continue;
    const unsigned* row = counts + slot * nc;
    unsigned long long sum = 0;
    unsigned best = 0;
    int arg = 0;
    for (int c = 0; c < nc; ++c) {
      const unsigned v = __ldg(row + c);
      sum += v;
      if (v > best) { best = v; arg = c; }     // strict: ties go to the lowest class
    }
    if (sum >= (unsigned long long)min_votes) out[i] = arg;
    return;
  }
}

static inline bool pow2(int64_t c) { return c > 0 && (c & (c - 1)) == 0; }

}  // namespace pcls

using namespace pcls;

#define SM_REQUIRE_SIZES(fn)                                                                                           \
  PCLS_REQUIRE(B >= 0 && total >= 0 && total < ((int64_t)1 << 31) && (B > 0 || total == 0),                           \
               fn ": bad sizes B=%d total=%lld (total must be < 2^31)", B, (long long)total);                          \
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= 32, fn ": num_classes %d not in [1,32]", num_classes);              \
  PCLS_REQUIRE(isfinite(voxel_size) && voxel_size > 0.0, fn ": voxel_size %g must be finite and > 0", voxel_size);    \
  PCLS_REQUIRE(pow2(capacity), fn ": capacity %lld is not a power of two", (long long)capacity);                       \
  PCLS_REQUIRE(table_keys != nullptr && table_counts != nullptr, fn ": table_keys / table_counts must not be NULL");   \
  PCLS_REQUIRE(offsets != nullptr && (B == 0 || poses != nullptr), fn ": offsets / poses must not be NULL");           \
  PCLS_REQUIRE(total == 0 || (points != nullptr && reinterpret_cast<uintptr_t>(points) % 16 == 0),                     \
               fn ": points must not be NULL and must be 16-byte aligned")

extern "C" int pcls_semantic_map_vote(const float* points, const int64_t* offsets, int B, int64_t total,
                                      const double* poses, double voxel_size, double min_range, double max_range,
                                      const int32_t* labels, int num_classes, int ignore_class, uint64_t* table_keys,
                                      uint32_t* table_counts, int64_t capacity, int64_t* state, pcls_stream stream) {
  SM_REQUIRE_SIZES("pcls_semantic_map_vote");
  PCLS_REQUIRE(ignore_class == -1 || (ignore_class >= 0 && ignore_class < num_classes),
               "pcls_semantic_map_vote: ignore_class %d must be -1 or in [0,%d)", ignore_class, num_classes);
  PCLS_REQUIRE(isfinite(min_range) && isfinite(max_range) && min_range >= 0.0 &&
               (max_range <= 0.0 || max_range >= min_range),
               "pcls_semantic_map_vote: range limits min %g max %g (need finite, 0 <= min, max <= 0 or max >= min)",
               min_range, max_range);
  PCLS_REQUIRE(state != nullptr, "pcls_semantic_map_vote: state must not be NULL");
  PCLS_REQUIRE(total == 0 || labels != nullptr, "pcls_semantic_map_vote: labels must not be NULL");
  if (total == 0) return PCLS_OK;
  const double min2 = min_range * min_range, max2 = max_range > 0.0 ? max_range * max_range : 0.0;
  map_vote_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
      points, offsets, B, total, poses, voxel_size, min2, max2, labels, num_classes, ignore_class,
      reinterpret_cast<unsigned long long*>(table_keys), table_counts, capacity, state);
  return check_launch("map_vote_kernel");
}

extern "C" int pcls_semantic_map_grow(const uint64_t* old_keys, const uint32_t* old_counts, int64_t old_capacity,
                                      int num_classes, uint64_t* new_keys, uint32_t* new_counts, int64_t new_capacity,
                                      int64_t* state, pcls_stream stream) {
  PCLS_REQUIRE(num_classes >= 1 && num_classes <= 32, "pcls_semantic_map_grow: num_classes %d not in [1,32]",
               num_classes);
  PCLS_REQUIRE(pow2(old_capacity) && pow2(new_capacity),
               "pcls_semantic_map_grow: capacities %lld -> %lld must be powers of two", (long long)old_capacity,
               (long long)new_capacity);
  PCLS_REQUIRE(old_keys != nullptr && old_counts != nullptr && new_keys != nullptr && new_counts != nullptr &&
               state != nullptr, "pcls_semantic_map_grow: tables and state must not be NULL");
  PCLS_REQUIRE((const void*)old_keys != (const void*)new_keys && (const void*)old_counts != (const void*)new_counts,
               "pcls_semantic_map_grow: the new table must not be the old one");
  cudaStream_t st = (cudaStream_t)stream;
  PCLS_CHECK_CUDA(cudaMemsetAsync(new_keys, 0xff, (size_t)new_capacity * sizeof(uint64_t), st));
  PCLS_CHECK_CUDA(cudaMemsetAsync(new_counts, 0, (size_t)new_capacity * num_classes * sizeof(uint32_t), st));
  map_grow_kernel<<<(unsigned)ceil_div(old_capacity, 256), 256, 0, st>>>(
      reinterpret_cast<const unsigned long long*>(old_keys), old_counts, old_capacity, num_classes,
      reinterpret_cast<unsigned long long*>(new_keys), new_counts, new_capacity, state);
  return check_launch("map_grow_kernel");
}

extern "C" int pcls_semantic_map_query(const float* points, const int64_t* offsets, int B, int64_t total,
                                       const double* poses, double voxel_size, const int32_t* labels_in,
                                       int num_classes, uint32_t keep_mask, int min_votes, const uint64_t* table_keys,
                                       const uint32_t* table_counts, int64_t capacity, int32_t* out_labels,
                                       pcls_stream stream) {
  SM_REQUIRE_SIZES("pcls_semantic_map_query");
  PCLS_REQUIRE(num_classes == 32 || (keep_mask >> num_classes) == 0,
               "pcls_semantic_map_query: keep_mask 0x%x names a class >= num_classes %d", keep_mask, num_classes);
  PCLS_REQUIRE(min_votes >= 1, "pcls_semantic_map_query: min_votes %d must be >= 1", min_votes);
  PCLS_REQUIRE(total == 0 || (labels_in != nullptr && out_labels != nullptr),
               "pcls_semantic_map_query: labels_in / out_labels must not be NULL");
  if (total == 0) return PCLS_OK;
  map_query_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, (cudaStream_t)stream>>>(
      points, offsets, B, total, poses, voxel_size, labels_in, num_classes, keep_mask, min_votes,
      reinterpret_cast<const unsigned long long*>(table_keys), table_counts, capacity, out_labels);
  return check_launch("map_query_kernel");
}
