// The logits layer (SqueezeSegV2 conv14, Darknet head: 3x3 conv to NUM_CLASS <= 20 channels, nets/SqueezeSegV2.py:276-282,
// nets/Darknet.py:255-260) fused with the segmentation head (softmax -> argmax -> depth-zero mask,
// nets/SegmentationNetwork.py:58-69), tcgen05 / TMEM / TMA, sm_100a.
//
// Why its own kernel.  In the generic implicit GEMM (conv_tc.cu) this layer issues 9 taps x Cin/16 MMAs of M128 x N32 x K16
// per 128-pixel tile.  Measured (tools/umma_bench.cu): an SS-mode tcgen05.mma costs max(N/2, 32 + N/4) cycles - below
// N = 128 it is bound by the shared-memory read of the A operand (128 rows x 32 bytes), not by the tensor pipe - so 36
// MMAs of N = 32 cost as much as 36 MMAs of N = 128, and the issuing warp was busy 92 % of the kernel (wait-cycle
// counters: 74 cycles per MMA, 2 880 cycles per tile against an HBM budget of 1 170).
//
// Horizontal tap packing.  The three horizontal taps (kx = 0,1,2) of one kernel row are stacked along N:
//     B[dh] = [ W[dh][0] ; W[dh][1] ; W[dh][2] ]          N = 3 x CS (CS = classes rounded up to 4), padded to 16
// and ONE MMA chain over the three kernel rows (3 x Cin/16 MMAs, 12 instead of 36 for Cin = 64) leaves in TMEM row x
//     T_kx[x] = sum_{dh,c} in[h+dh-1, x, c] * W[dh][kx][c]              for the 128 INPUT pixels x of the tile.
// The output pixel w is T_0[w-1] + T_1[w] + T_2[w+1]: a +-1 shift across TMEM lanes, done in the epilogue with two warp
// shuffles per class (the two lanes at the warp boundary go through shared memory).  A tile therefore covers input
// pixels w0-1 .. w0+126 (one TMA box of 128 rows per kernel row, zero-filled outside the image = SAME padding) and
// produces the 126 output pixels w0 .. w0+125.
//
// Warp roles as in conv_tc.cu (576 threads): warp 0 TMA producer, warp 1 MMA issuer, warps 2-17 four epilogue groups that
// take tiles round-robin.  The epilogue copies the accumulator row to registers, releases the TMEM buffer at once, and then
// runs bias -> shift-sum (a lane rotation, the boundary lanes' unread rows swapped through smem) -> softmax (SFU ex2) ->
// argmax over the rounded probabilities -> mask -> stores; every warp stages its pixels x classes block in shared memory
// in output layout and ships it with one bulk copy.
//
// Pipeline.  ONE stage = all 3 x Cin/KC input tiles of an output tile behind one full / empty mbarrier pair (3 stages of
// 48 KB for Cin = 64): the issuing thread makes two barrier waits and two tcgen05.commit per tile.  With a stage per
// input tile (four waits, four commits) the kernel took 0.210 instead of 0.178 ms at batch 32 - its issuer never waited
// FOR anything, it paid the round-trip latency of the waits and commits themselves (DESIGN.md section 6, step 27).
#include "tc_ptx.cuh"

#include <cstring>
#include <vector>

namespace pcls {

constexpr int HD_NG = 4;                        // epilogue warp-groups (4 warps each); tiles are dealt round-robin
// -DPCLS_HEAD_ISSUERS=2 (experimental, NOT validated on hardware yet - DESIGN.md section 6, step 27): a second MMA-issuing
// warp (the last warp of the CTA); the two take alternate tiles so that their barrier / commit round trips overlap.  The
// stage ring is then forced to an EVEN length: tile sequence number s lives in stage s % S, so with S even issuer i only
// ever touches stages = i (mod 2) and accumulators = i (mod 2) - it has consumed the previous round of every barrier it
// waits on itself.  (With three stages the issuers shared stages, the faster one could reach a stage a full ring round
// ahead of the slower one, the parity wait returned on the stale phase: launch failure at batch 32.)
#ifndef PCLS_HEAD_ISSUERS
#define PCLS_HEAD_ISSUERS 1
#endif
#if PCLS_HEAD_ISSUERS == 2
constexpr int HD_ISSUER2 = 2 + 4 * HD_NG;
#endif
constexpr int HD_THREADS = 64 + 128 * HD_NG + 32 * (PCLS_HEAD_ISSUERS - 1);
constexpr int HD_TILE = 126;   // output pixels per tile (128 input pixels incl. the one-pixel halo on both sides)

struct HeadParams {
  int pdl_early;               // trigger the dependent grid at the start (common.cuh)
  int H, W, n_wt;
  int kchunks;                 // Cin / KC
  int N, cout;                 // MMA N (multiple of 16 >= 3 CS), classes
  int stages, a_bytes, b_tile_bytes, bres_bytes;
  uint32_t idesc, desc_hi, tmem_cols;
  int n_acc;
  const float* bias;
  float slope;                 // activation as max(v, v * slope): 1 = none
  int stg_warp_floats;         // per-warp output staging (floats): 32 x cout when cout % 4 == 0, else 32 x 33
  int head, none_index;        // head = 1: softmax / argmax / mask; 0: logits only (written to `logits`)
  const uint8_t* mask;
  float* probs;
  int32_t* preds;
  float* logits;
};

template <typename T, int KC, int CS>
__global__ void __launch_bounds__(HD_THREADS, 1)
conv_head_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ HeadParams p, const int num_tiles) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = smem_u32(smem_raw);
  const uint32_t smem_base = (smem0 + 1023u) & ~1023u;
  const int S = p.stages;
  const uint32_t a_bytes = (uint32_t)p.a_bytes, b_tile_bytes = (uint32_t)p.b_tile_bytes;
  const uint32_t stage_bytes = (uint32_t)(3 * p.kchunks) * a_bytes;   // one stage = the 3 x kchunks input tiles of an output tile
  const uint32_t bres_base = smem_base + (uint32_t)S * stage_bytes;            // resident weights [3][kchunks] tiles
  const uint32_t stg_base = bres_base + (uint32_t)p.bres_bytes;            // [4 HD_NG warps][stg_warp_floats] f32 output staging
  const uint32_t xch_base = stg_base + (uint32_t)(4 * HD_NG * p.stg_warp_floats) * 4u;   // [groups][2 buffers][4 quarters][2 CS] f32
  const uint32_t bar_base = xch_base + (uint32_t)HD_NG * 2u * 4u * 2u * (uint32_t)CS * 4u;
#define FULL_BAR(s) (bar_base + 8u * (uint32_t)(s))
#define EMPTY_BAR(s) (bar_base + 8u * (uint32_t)(S + (s)))
#define TFULL_BAR(a) (bar_base + 8u * (uint32_t)(2 * S + (a)))
#define TEMPTY_BAR(a) (bar_base + 8u * (uint32_t)(2 * S + 8 + (a)))
#define BRES_BAR (bar_base + 8u * (uint32_t)(2 * S + 16))
  const uint32_t tmem_slot = bar_base + 8u * (uint32_t)(2 * S + 17);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem0));
  float* bias_s = reinterpret_cast<float*>(smem_raw + (((tmem_slot + 16u + 15u) & ~15u) - smem0));   // [CS], 16-byte aligned
  // classes >= cout (padding up to CS) get a bias of -inf: they drop out of max / softmax / argmax without range checks
  if (threadIdx.x < CS) bias_s[threadIdx.x] = (int)threadIdx.x < p.cout ? p.bias[threadIdx.x] : -INFINITY;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    for (int s = 0; s < S; ++s) { mbar_init(FULL_BAR(s), 1); mbar_init(EMPTY_BAR(s), 1); }
    for (int a = 0; a < 8; ++a) { mbar_init(TFULL_BAR(a), 1); mbar_init(TEMPTY_BAR(a), 4); }
    mbar_init(BRES_BAR, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const int n_wt = p.n_wt, H = p.H, W = p.W, kchunks = p.kchunks;
  const uint32_t N = (uint32_t)p.N;
  pdl_trigger(p.pdl_early);     // PDL (common.cuh): prologue and weight loads overlap the tail of the layer in front
  if (warp != 0) pdl_wait();

  if (warp == 0) {
    // ===================== TMA producer =====================
    mbar_arrive_expect_tx_elect(BRES_BAR, (uint32_t)(3 * kchunks) * b_tile_bytes);
    for (int g = 0; g < 3; ++g)
      for (int kc = 0; kc < kchunks; ++kc)
        tma_load_3d_elect(bres_base + (uint32_t)(g * kchunks + kc) * b_tile_bytes, &map_b, BRES_BAR, kc * KC, 0, g);
    pdl_wait();
    int stage = 0;
    uint32_t phase = 0;
    // One pipeline stage = ALL input tiles of an output tile (3 rows x kchunks, 16 KB each) behind ONE full / empty
    // barrier pair: the MMA issuer pays two barrier waits and two commits per tile instead of four and four (its spin
    // counters never show it waiting, the tensor pipe is 25 % busy and trimming its instruction stream changed nothing:
    // what it spends its time on is the latency of the mbarrier / commit round trips themselves).
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int wt = tile % n_wt, h = (tile / n_wt) % H, b = tile / (n_wt * H);
      const int ww = wt * HD_TILE - 1;
      mbar_wait(EMPTY_BAR(stage), phase ^ 1u);
      const uint32_t fb = FULL_BAR(stage);
      mbar_arrive_expect_tx_elect(fb, (uint32_t)(3 * kchunks) * 128u * KC * 2u);
      uint32_t dst = smem_base + (uint32_t)stage * stage_bytes;
      for (int g = 0; g < 3; ++g)
        for (int kc = 0; kc < kchunks; ++kc) {
          tma_load_4d_elect(dst, &map_a, fb, kc * KC, ww, h + g - 1, b);
          dst += a_bytes;
        }
      if (++stage == S) { stage = 0; phase ^= 1u; }
    }
#if PCLS_HEAD_ISSUERS == 2
  } else if (warp == 1 || warp == HD_ISSUER2) {
    // ===================== MMA issuers (two warps, alternate tiles; see PCLS_HEAD_ISSUERS above) =====================
    const uint32_t desc_hi = p.desc_hi, idesc = p.idesc, n_acc = (uint32_t)p.n_acc, acc_shift2 = 31u - (uint32_t)__clz(p.n_acc);
    const int k_iters = 3 * kchunks;
    const uint32_t iw = warp == 1 ? 0u : 1u;
    int stage = (int)iw;                 // S is even and >= 2
    uint32_t phase = 0, seq = iw;
    mbar_wait(BRES_BAR, 0u);
    for (long long tile = (long long)blockIdx.x + (long long)iw * gridDim.x; tile < num_tiles; tile += 2LL * gridDim.x, seq += 2u) {
      const uint32_t acc = seq & (n_acc - 1u), acc_phase = (seq >> acc_shift2) & 1u;
      mbar_wait(TEMPTY_BAR(acc), acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * N;
      uint32_t b_addr = bres_base, accumulate = 0u;
      mbar_wait(FULL_BAR(stage), phase);
      tc_fence_after();
      uint32_t a_addr = smem_base + (uint32_t)stage * stage_bytes;
      for (int k = 0; k < k_iters; ++k) {
        umma_f16_ksteps_elect<KC / 16>(d_tmem, ((a_addr >> 4) & 0x3FFFu) | 0x10000u, desc_hi, ((b_addr >> 4) & 0x3FFFu) | 0x10000u,
                                       desc_hi, idesc, accumulate);
        accumulate = 1u;
        a_addr += a_bytes;
        b_addr += b_tile_bytes;
      }
      umma_commit_elect(EMPTY_BAR(stage));
      stage += 2;
      if (stage >= S) { stage -= S; phase ^= 1u; }
      umma_commit_elect(TFULL_BAR(acc));
    }
#else
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t desc_hi = p.desc_hi, idesc = p.idesc, n_acc = (uint32_t)p.n_acc;
    const int k_iters = 3 * kchunks;
    int stage = 0;
    uint32_t phase = 0, acc = 0, acc_phase = 0;
    mbar_wait(BRES_BAR, 0u);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(TEMPTY_BAR(acc), acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * N;
      uint32_t b_addr = bres_base, accumulate = 0u;
      mbar_wait(FULL_BAR(stage), phase);
      tc_fence_after();
      uint32_t a_addr = smem_base + (uint32_t)stage * stage_bytes;
      for (int k = 0; k < k_iters; ++k) {
        // the KC / 16 K steps of this chunk behind one elect (tc_ptx.cuh)
        umma_f16_ksteps_elect<KC / 16>(d_tmem, ((a_addr >> 4) & 0x3FFFu) | 0x10000u, desc_hi, ((b_addr >> 4) & 0x3FFFu) | 0x10000u,
                                       desc_hi, idesc, accumulate);
        accumulate = 1u;
        a_addr += a_bytes;
        b_addr += b_tile_bytes;
      }
      umma_commit_elect(EMPTY_BAR(stage));   // the stage is free once these MMAs have read it
      if (++stage == S) { stage = 0; phase ^= 1u; }
      umma_commit_elect(TFULL_BAR(acc));
      if (++acc == n_acc) { acc = 0; acc_phase ^= 1u; }
    }
#endif
  } else {
    // ===================== epilogue: two groups of four warps, alternate tiles =====================
    const int ew = warp - 2, grp = ew >> 2, q = warp & 3;   // q = TMEM lane quarter this warp may read
    const int r = q * 32 + lane;                            // accumulator row = input pixel w0 - 1 + r
    const uint32_t n_acc = (uint32_t)p.n_acc, acc_shift = 31u - (uint32_t)__clz(p.n_acc);   // (a power of two)
    const int cout = p.cout;
    const float slope = p.slope;
    float* const stg = reinterpret_cast<float*>(smem_raw + (stg_base - smem0)) + ew * p.stg_warp_floats;
    float* const xch = reinterpret_cast<float*>(smem_raw + (xch_base - smem0)) + grp * (2 * 4 * 2 * CS);
    uint32_t cnt = 0;
    // this thread's output pixel of the group's next tile (r = 0 and r = 127 are halo rows, not outputs).  The group's tiles
    // advance by a constant stride (HD_NG * gridDim.x): the (column tile, row, frame) coordinates are kept incrementally -
    // three integer divisions per tile were ~100 of the ~820 instructions an epilogue warp spends per tile.
    const long long stride_ll = (long long)HD_NG * gridDim.x;
    const int s_wt = (int)(stride_ll % n_wt), s_h = (int)((stride_ll / n_wt) % H), s_b = (int)(stride_ll / ((long long)n_wt * H));
    long long t_ll = (long long)blockIdx.x + (long long)grp * gridDim.x;
    int c_wt = (int)(t_ll % n_wt), c_h = (int)((t_ll / n_wt) % H), c_b = (int)(t_ll / ((long long)n_wt * H));
    auto locate = [&](int64_t& pix, bool& valid) -> bool {
      if (t_ll >= num_tiles) { pix = 0; valid = false; return false; }
      const int w = c_wt * HD_TILE - 1 + r;
      valid = r >= 1 && r <= HD_TILE && w < W;
      pix = ((int64_t)c_b * H + c_h) * W + w;
      t_ll += stride_ll;
      c_wt += s_wt;
      if (c_wt >= n_wt) { c_wt -= n_wt; ++c_h; }
      c_h += s_h;
      if (c_h >= H) { c_h -= H; ++c_b; }
      c_b += s_b;
      return true;
    };
    int64_t pix, pix_n;
    bool valid, valid_n;
    uint32_t tl = (uint32_t)grp;
    bool have = locate(pix, valid);
    uint32_t head_mask = (have && p.head && valid) ? p.mask[pix] : 1u;
    while (have) {
      // the NEXT tile's mask byte travels during this tile's work (its latency was 10 % of the kernel's stall samples)
      const bool have_n = locate(pix_n, valid_n);
      const uint32_t head_mask_n = (have_n && p.head && valid_n) ? p.mask[pix_n] : 1u;
      const uint32_t acc = tl & (n_acc - 1u), acc_parity = (tl >> acc_shift) & 1u;
      mbar_wait(TFULL_BAR(acc), acc_parity);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + acc * N;
      uint32_t v0[32], v1[32];            // accumulator columns [0, 32) and [32, 64); V(i) resolves statically after unrolling
#define V(i) ((i) < 32 ? v0[(i) & 31] : v1[((i) - 32) & 31])
      tmem_ld32(t_row, v0);
      if (3 * CS > 48) {
        tmem_ld32(t_row + 32u, v1);
      } else if (3 * CS > 32) {
        uint32_t t16[16];
        tmem_ld16(t_row + 32u, t16);
#pragma unroll
        for (int j = 0; j < 16; ++j) { v1[j] = t16[j]; v1[16 + j] = 0u; }
      }
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(TEMPTY_BAR(acc));           // accumulator free: everything below runs from registers

      // ---- out[w] = T0[w-1] + T1[w] + T2[w+1]: +-1 lane shuffles; the lanes at the warp boundary go through smem ----
      float* const xb = xch + (cnt & 1u) * (4 * 2 * CS);
      ++cnt;
      if (lane == 31) {
#pragma unroll
        for (int c = 0; c < CS; c += 4)
          *reinterpret_cast<float4*>(xb + q * 2 * CS + c) = make_float4(__uint_as_float(V(c)), __uint_as_float(V(c + 1)),
                                                                        __uint_as_float(V(c + 2)), __uint_as_float(V(c + 3)));
      }
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < CS; c += 4)
          *reinterpret_cast<float4*>(xb + q * 2 * CS + CS + c) = make_float4(__uint_as_float(V(2 * CS + c)), __uint_as_float(V(2 * CS + c + 1)),
                                                                             __uint_as_float(V(2 * CS + c + 2)), __uint_as_float(V(2 * CS + c + 3)));
      }
      group_barrier(1 + grp);   // (also orders the reuse of this exchange buffer two tiles later)
      // Lane 31's own T0 row has no reader inside the warp (it went to the next quarter through smem) and neither has
      // lane 0's T2 row: they are REPLACED by the neighbouring quarter's rows, and a rotation by one lane then hands every
      // lane - the boundary lanes included - the right neighbour value: no edge selects, no fix-up adds (-80 of ~820
      // instructions per warp and tile).  Quarter 0 / lane 0 and quarter 3 / lane 31 are the halo rows r = 0 / 127: not outputs.
      if (lane == 31 && q > 0) {
#pragma unroll
        for (int c = 0; c < CS; c += 4) {
          const float4 t = *reinterpret_cast<const float4*>(xb + (q - 1) * 2 * CS + c);
          V(c) = __float_as_uint(t.x); V(c + 1) = __float_as_uint(t.y); V(c + 2) = __float_as_uint(t.z); V(c + 3) = __float_as_uint(t.w);
        }
      }
      if (lane == 0 && q < 3) {
#pragma unroll
        for (int c = 0; c < CS; c += 4) {
          const float4 t = *reinterpret_cast<const float4*>(xb + (q + 1) * 2 * CS + CS + c);
          V(2 * CS + c) = __float_as_uint(t.x); V(2 * CS + c + 1) = __float_as_uint(t.y);
          V(2 * CS + c + 2) = __float_as_uint(t.z); V(2 * CS + c + 3) = __float_as_uint(t.w);
        }
      }
      const int lane_l = (lane + 31) & 31, lane_r = (lane + 1) & 31;
      float lg[CS];
#pragma unroll
      for (int c = 0; c < CS; ++c) {
        const float left = __shfl_sync(0xffffffffu, __uint_as_float(V(c)), lane_l);             // T0 of row r-1
        const float right = __shfl_sync(0xffffffffu, __uint_as_float(V(2 * CS + c)), lane_r);  // T2 of row r+1
        lg[c] = __uint_as_float(V(CS + c)) + left + right;
      }
      // bias (-inf for the padding classes), activation (none for conv14 / head: slope 1)
#pragma unroll
      for (int c = 0; c < CS; c += 4) {
        const float4 bv = *reinterpret_cast<const float4*>(bias_s + c);
        lg[c] += bv.x; lg[c + 1] += bv.y; lg[c + 2] += bv.z; lg[c + 3] += bv.w;
      }
      if (slope != 1.0f) {
#pragma unroll
        for (int c = 0; c < CS; ++c) lg[c] = fmaxf(lg[c], lg[c] * slope);
      }

      const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
      const int n_valid = __popc(vmask), first = vmask ? __ffs(vmask) - 1 : 0;   // valid lanes are consecutive
      const int64_t pix0 = __shfl_sync(0xffffffffu, pix, first);
      auto write_rows = [&](float* dst) {                      // lg[] of the valid pixels -> dst[pix0*cout ..] coalesced
        if ((cout & 3) == 0) {
          if (lane == 0) bulk_wait_read0();                    // the previous copy has finished reading the staging rows
          __syncwarp();
          if (valid) {
#pragma unroll
            for (int c = 0; c < CS; c += 4)
              if (c < cout) *reinterpret_cast<float4*>(stg + (lane - first) * cout + c) = make_float4(lg[c], lg[c + 1], lg[c + 2], lg[c + 3]);
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0 && n_valid > 0) {
            bulk_store_1d(dst + pix0 * cout, smem_u32(stg), (uint32_t)(n_valid * cout * 4));
            bulk_commit();
          }
          return;
        }
        __syncwarp();
        if (valid) {
#pragma unroll
          for (int c = 0; c < CS; ++c) if (c < cout) stg[(lane - first) * 33 + c] = lg[c];
        }
        __syncwarp();
        const int n_el = n_valid * cout;
        int px = lane / cout, cc = lane - px * cout;            // (pixel, class) of element `lane`, advanced by 32
        const int dpx = 32 / cout, dcc = 32 - dpx * cout;
        for (int e = lane; e < n_el; e += 32) {
          dst[pix0 * cout + e] = stg[px * 33 + cc];
          px += dpx; cc += dcc;
          if (cc >= cout) { cc -= cout; ++px; }
        }
        __syncwarp();
      };
      if (p.logits) write_rows(p.logits);
      if (p.head) {
        // softmax with SFU exponentials and one reciprocal, argmax over the rounded probabilities, first index on ties
        float mx = lg[0];
#pragma unroll
        for (int c = 0; c < CS; c += 4) mx = fmaxf(fmaxf(mx, fmaxf(lg[c], lg[c + 1])), fmaxf(lg[c + 2], lg[c + 3]));
        float sum = 0.0f;
        const float mxl = -mx * 1.4426950408889634f;
#pragma unroll
        for (int c = 0; c < CS; ++c) { lg[c] = ex2_ftz(fmaf(lg[c], 1.4426950408889634f, mxl)); sum += lg[c]; }
        const float inv = __fdividef(1.0f, sum);
        int best = 0;
        float bp = -1.0f;
#pragma unroll
        for (int c = 0; c < CS; ++c) { lg[c] *= inv; if (lg[c] > bp) { bp = lg[c]; best = c; } }
        if (valid) {
          if (head_mask == 0) best = p.none_index;
          p.preds[pix] = best;
        }
        if (p.probs) write_rows(p.probs);
      }
      tl += HD_NG; have = have_n; pix = pix_n; valid = valid_n; head_mask = head_mask_n;
    }
    if (lane == 0) bulk_wait_all();   // the staging rows must outlive the last bulk copies
  }

  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
#undef V
#undef FULL_BAR
#undef EMPTY_BAR
#undef TFULL_BAR
#undef TEMPTY_BAR
#undef BRES_BAR
}

struct HeadPlan {
  CUtensorMap map_a, map_b;
  HeadParams prm;
  size_t smem_bytes;
  void* w_dev = nullptr;
  int KC, CS, is_bf16;
};

typedef void (*HeadKernelFn)(const CUtensorMap, const CUtensorMap, const HeadParams, const int);
template <typename T>
static HeadKernelFn head_kernel_for_t(int KC, int CS) {
  if (KC == 64) return CS == 8 ? conv_head_kernel<T, 64, 8> : CS == 12 ? conv_head_kernel<T, 64, 12> : CS == 16 ? conv_head_kernel<T, 64, 16> : conv_head_kernel<T, 64, 20>;
  return CS == 8 ? conv_head_kernel<T, 32, 8> : CS == 12 ? conv_head_kernel<T, 32, 12> : CS == 16 ? conv_head_kernel<T, 32, 16> : conv_head_kernel<T, 32, 20>;
}
static HeadKernelFn head_kernel_for(int KC, int CS, int bf16) {
  return bf16 ? head_kernel_for_t<__nv_bfloat16>(KC, CS) : head_kernel_for_t<__half>(KC, CS);
}

// Plans the logits layer for conv_head_kernel when its shape allows: 3x3 stride-1 conv from a tensor with 32 k channels
// to <= 20 float32 logits, no residuals.  Returns PCLS_OK with L.hp == nullptr when the layer does not qualify.
int Net::head_plan_layer(ConvLayer& L) {
  L.hp = nullptr;
  const ConvParams& cp = L.p;
  if (!cp.out_f32 || cp.mode != MODE_3x3_S1 || L.pair_view || L.res0 >= 0 || L.res1 >= 0) return PCLS_OK;
  if (cp.cin_pad % 32 != 0 || cp.cin_pad > cp.in_channels || cp.cout > 20 || cp.out_coff != 0 || cp.out_channels != cp.cout) return PCLS_OK;
  if (cp.Win != cp.Wout || cp.Wout < 64) return PCLS_OK;
  const bool bf16 = precision == PCLS_BF16;
  HeadPlan* plan = new HeadPlan();
  HeadParams& q = plan->prm;
  memset(&q, 0, sizeof(q));
  const int KC = cp.cin_pad % 64 == 0 ? 64 : 32;
  int CS = (cp.cout + 3) / 4 * 4;
  if (CS < 8) CS = 8;
  plan->KC = KC; plan->CS = CS; plan->is_bf16 = bf16 ? 1 : 0;
  q.H = cp.H; q.W = cp.Wout; q.n_wt = (cp.Wout + HD_TILE - 1) / HD_TILE;
  q.kchunks = cp.cin_pad / KC;
  q.N = (3 * CS + 15) / 16 * 16;
  q.cout = cp.cout;
  q.a_bytes = 128 * KC * 2;
  q.b_tile_bytes = q.N * KC * 2;
  q.bres_bytes = (3 * q.kchunks * q.b_tile_bytes + 1023) / 1024 * 1024;
  const int swz = KC * 2;
  const uint32_t layout = swz == 128 ? 2u : 4u;
  q.desc_hi = ((uint32_t)(8 * swz) >> 4) | (1u << 14) | (layout << 29);
  q.idesc = (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | ((uint32_t)(q.N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  q.n_acc = 8;
  while (q.n_acc * q.N > 512) q.n_acc /= 2;
  uint32_t cols = 32;
  while (cols < (uint32_t)(q.n_acc * q.N)) cols <<= 1;
  q.tmem_cols = cols;
  q.bias = cp.bias;
  q.slope = cp.act == PCLS_ACT_RELU ? 0.0f : (cp.act == PCLS_ACT_LEAKY ? 0.1f : 1.0f);
  q.stg_warp_floats = (cp.cout % 4 == 0) ? 32 * cp.cout : 32 * 33;
  const int fixed = q.bres_bytes + 4 * HD_NG * q.stg_warp_floats * 4 + HD_NG * 2 * 4 * 2 * CS * 4 + 1024 /*alignment*/ + 512 /*barriers, slot, bias*/;
  const int stage_bytes = 3 * q.kchunks * q.a_bytes;   // a stage holds every input tile of one output tile
  int stages = (227 * 1024 - fixed) / stage_bytes;
  if (stages > 4) stages = 4;
#if PCLS_HEAD_ISSUERS == 2
  stages -= stages % 2;   // each issuer owns the stages of its parity
  if (q.n_acc < 2) { delete plan; return PCLS_OK; }
#endif
  if (stages < 2) { delete plan; return PCLS_OK; }
  q.stages = stages;
  plan->smem_bytes = (size_t)stages * stage_bytes + fixed;

  // weights: [kernel row dh][n = kx * CS + class][ci], K-major, 16-bit
  std::vector<uint16_t> packed((size_t)3 * q.N * cp.cin_pad, 0);
  for (int dh = 0; dh < 3; ++dh)
    for (int kx = 0; kx < 3; ++kx)
      for (int c = 0; c < cp.cout; ++c)
        for (int ci = 0; ci < cp.cin_pad; ++ci) {
          const float w = L.w_f32[((size_t)(dh * 3 + kx) * cp.cout_pad + c) * cp.cin_pad + ci];
          uint16_t bits;
          if (bf16) { __nv_bfloat16 hv = __float2bfloat16_rn(w); memcpy(&bits, &hv, 2); }
          else { __half hv = __float2half_rn(w); memcpy(&bits, &hv, 2); }
          packed[((size_t)dh * q.N + kx * CS + c) * cp.cin_pad + ci] = bits;
        }
  if (cudaMalloc(&plan->w_dev, packed.size() * 2) != cudaSuccess) { delete plan; set_error("head plan: cudaMalloc failed"); return PCLS_ERR_CUDA; }
  if (cudaMemcpy(plan->w_dev, packed.data(), packed.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaFree(plan->w_dev); delete plan; set_error("head plan: weight upload failed"); return PCLS_ERR_CUDA;
  }
  int rc;
  {
    char* a_base = (char*)tensor_ptr(L.in, frames_per_pass);
    const uint64_t C = (uint64_t)cp.in_channels, Wi = (uint64_t)cp.Win, Hh = (uint64_t)cp.H, F = (uint64_t)frames_per_pass;
    const uint64_t dims[4] = {C, Wi, Hh, F};
    const uint64_t str[3] = {C * 2, Wi * C * 2, Hh * Wi * C * 2};
    const uint32_t box[4] = {(uint32_t)KC, 128u, 1u, 1u};
    rc = make_map(&plan->map_a, bf16, a_base, 4, dims, str, box, swz);
  }
  if (rc == PCLS_OK) {
    const uint64_t dims[3] = {(uint64_t)cp.cin_pad, (uint64_t)q.N, 3};
    const uint64_t str[2] = {(uint64_t)cp.cin_pad * 2, (uint64_t)cp.cin_pad * q.N * 2};
    const uint32_t box[3] = {(uint32_t)KC, (uint32_t)q.N, 1u};
    rc = make_map(&plan->map_b, bf16, plan->w_dev, 3, dims, str, box, swz);
  }
  if (rc) { cudaFree(plan->w_dev); delete plan; return rc; }
  cudaError_t e = cudaFuncSetAttribute(head_kernel_for(KC, CS, bf16 ? 1 : 0), cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
  if (e != cudaSuccess) { cudaFree(plan->w_dev); delete plan; set_error("head plan: %s", cudaGetErrorString(e)); return PCLS_ERR_CUDA; }
  L.hp = plan;
  return PCLS_OK;
}

int Net::head_launch(ConvLayer& L, const ConvParams& p, int nb, cudaStream_t s) {
  HeadPlan* plan = L.hp;
  HeadParams prm = plan->prm;
  prm.head = head_args.head;
  prm.none_index = head_args.none_index; prm.mask = head_args.mask;
  prm.pdl_early = pdl_early_now;
  prm.preds = head_args.preds;
  prm.probs = head_args.head ? head_args.probs : nullptr;
  // fused head: logits travel to HBM only when the caller asks for them; unfused: this layer's output IS the logits tensor
  prm.logits = head_args.head ? head_args.logits : reinterpret_cast<float*>(p.out);
  const int num_tiles = prm.n_wt * prm.H * nb;
  if (num_tiles == 0) return PCLS_OK;
  const int grid = num_tiles < sm_count() ? num_tiles : sm_count();
  PCLS_CHECK_CUDA(launch_pdl(head_kernel_for(plan->KC, plan->CS, plan->is_bf16), dim3(grid), dim3(HD_THREADS), plan->smem_bytes, s,
                             plan->map_a, plan->map_b, prm, num_tiles));
  return check_launch("conv_head_kernel");
}

void Net::head_release(ConvLayer& L) {
  if (L.hp) { if (L.hp->w_dev) cudaFree(L.hp->w_dev); delete L.hp; L.hp = nullptr; }
}

}  // namespace pcls
