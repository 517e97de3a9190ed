// tcgen05 / TMEM / TMA implicit-GEMM convolution for sm_100a.
//
// One persistent, warp-specialised kernel runs every convolution flavour of SqueezeSegV2 and Darknet whose channel
// counts fit UMMA tiles (3x3 s1, 3x3 s[1,2], 1x1, transposed [1,4] s[1,2]):
//
//   GEMM view      M = 128 output pixels (BH rows x BW columns of one frame), N = BN output channels,
//                  K = taps x Cin, walked as (tap, KC-channel chunk) iterations.
//   A operand      NHWC activations.  For tap (dh, dw) the tile is the SAME box shifted by (dh, dw): one TMA
//                  tiled load per iteration from a 4-D map (C, W, H, B); out-of-bounds rows/columns are zero-filled
//                  by TMA, which IS the SAME padding (no im2col buffer, no halo code).  The stride-2 convolutions read a
//                  5-D view (C, 2, W/2, H, B) of the same buffer: TF's asymmetric SAME padding for even W (0 left /
//                  1 right) makes tap kx land on (parity kx&1, pair wo + (kx>>1)), never left of the image.
//   A variants     3x3 stride-1 layers >= 128 pixels wide: ONE 130-pixel tile (1-pixel halo) per input row serves the three
//                  horizontal taps, the UMMA descriptor starts 0 / 1 / 2 rows into it.  Inputs with 16 / 32 channels:
//                  G = 4 / 2 adjacent pixels form one 128-byte row (pixel-group view) and the MMAs are issued banded.
//   B operand      folded weights packed [tap][Cout][Cin] (K-major); resident in smem for the whole kernel when the
//                  layer fits, else one TMA load per iteration.  Split-N: output channels [0, n1) that are zero outside
//                  the centre tap (merged Fire expand1x1 || expand3x3) are skipped by the eight outer taps.
//   MMA            tcgen05.mma.cta_group::1.kind::f16, M=128 x N=BN x K=16, fp32 accumulators in TMEM, 2-8 accumulator
//                  buffers (n_acc x BN <= 512 columns) so the epilogue of tile i overlaps the MMAs of tiles i+1...
//   epilogue       tcgen05.ld x32 -> +bias (BatchNorm folded) -> ReLU / LeakyReLU -> + residual(s) -> 16-bit NHWC output at
//                  a channel offset (tf.concat): swizzled smem tile + TMA bulk tensor store when the N tile is a multiple
//                  of 64 channels (residual blocks are TMA-loaded into the same staging buffers one block ahead), else
//                  16-byte stores; or float32 logits with the segmentation head (softmax / argmax / mask) fused.
//                  The transposed convolution runs as ONE 3-tap GEMM with N = 2 Cout (net.cu: build_deconv_row3); the
//                  two-phase form (even / odd output columns) remains for shapes that form rejects.
//
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer (both run warp-uniformly, the
// instruction is predicated on elect.sync), warps 2-9 = two epilogue groups that alternate tiles (TMEM lane quarter =
// warp_id % 4).  mbarrier rings: full/empty per smem stage, tmem_full/tmem_empty per accumulator.
#include "tc_ptx.cuh"

#include <cstring>

namespace pcls {

// ---------------------------------------------------------------------------------------------------------------
// kernel parameters
// ---------------------------------------------------------------------------------------------------------------
constexpr int TC_MAX_TAPS = 9;
// Epilogue warp-groups (4 warps each; tiles are dealt round-robin).  Kernels with residual adds need ~166 registers per
// thread: two groups (320 threads).  Kernels without (bias pre-loaded, ReLU in the conversion) need ~125 and could run
// three (448 threads) - measured slower on SqueezeSegV2 (3.83 vs 3.71 ms): the third group's staging buffers cost the
// layers with resident weights their pipeline stages.
constexpr int TC_NG = 2;
constexpr int TC_THREADS = 64 + 128 * TC_NG;   // warp 0 TMA producer, warp 1 MMA issuer, then the groups

struct TcParams {
  int pdl_early;              // trigger the dependent grid at the start (common.cuh)
  // tile geometry
  int BW, BH, bw_shift;       // BW * BH = 128, BW = 1 << bw_shift
  int n_wt, n_ht, n_nt, n_phase, num_tiles;
  int Hgrid, Wgrid;           // extent of the tiled pixel grid (output grid; input grid for the transposed conv)
  int out_wmul;               // output column = w * out_wmul + phase
  int Wout;
  // K walk: per tile, n_groups A loads per K chunk; each A tile feeds `sub` tap MMAs that start `sub_row[s]` rows into it
  int n_groups, sub;
  int kchunks;                // cin_pad / KC
  int ksteps;                 // UMMA K steps (16 channels) worth issuing per K chunk: KC / 16, fewer when the chunk's tail is
                              // zero padding (48 channels stored with a 64-channel stride: 3).  Host-side: selects the kernel.
  int KC, BN;
  int grp_dh[2][TC_MAX_TAPS], grp_dw[2][TC_MAX_TAPS], grp_par[2][TC_MAX_TAPS];  // TMA coordinate offsets of the A box
  int grp_w[2][TC_MAX_TAPS][3];                                                  // weight tap index per (group, sub)
  int sub_row[3];
  int a_is_5d;
  int a_rows;                 // rows of the A box: 128, or 130 with the one-pixel halo on both sides
  int b_resident;             // 1: every weight tile of the layer is loaded into smem once per CTA
  // pipeline
  int stages, a_bytes, b_tile_bytes, bres_bytes;
  uint32_t idesc, desc_hi;    // instruction descriptor; high 32 bits of the smem matrix descriptors
  uint32_t tmem_cols;
  int n_acc;                  // TMEM accumulator buffers (power of two, n_acc * BN <= 512)
  // TMA-store epilogue: output staged in smem in blocks of `cbw` channels (128 rows x cbw), two buffers per group
  int tma_store, cbw, c_is_5d, c_stage_bytes;
  // pixel-group view (G > 1): an A row holds G adjacent pixels x Cin channels; accumulator columns [p*cout_blk, ..) belong
  // to pixel p of the group.  cout_blk = 1 << 30 when G == 1.
  int G, cout_blk, cout_blk_shift;
  int res_smem;               // RES kernels: 1 = residual0 staged through smem with cp.async, 0 = per-chunk LDG
  int res_tma;                // RES kernels with the TMA-store epilogue: residual0 blocks are TMA-loaded INTO the output
                              // staging buffers one block ahead (three buffers per group), added in place, stored by TMA
  int n_cbuf;                 // output staging buffers per epilogue group (2, or 3 with res_tma)
  // split-N (merged Fire expand1x1 || expand3x3, nets/SqueezeSegV2.py:30-40): output channels [0, n1) have a non-zero
  // kernel only at the centre tap.  The other eight taps then load and multiply only the weight rows [n1, BN).
  int n1, b_small_bytes, bres_tx;
  uint32_t idesc_small, idesc_lo;
  // N-split across CTAs (nsplit = 1): the layer's N is cut into n_nt tiles of BN channels and the grid is a multiple of n_nt,
  // so a CTA only ever sees ONE N tile (tile % n_nt == blockIdx.x % n_nt) and keeps that tile's weights resident - for
  // layers whose whole weight set does not fit in smem (the A tiles are read n_nt times, from L2).  With perm = 1 the
  // weight / bias rows were permuted so that every N tile holds a slice of both halves of a merged Fire expand
  // (centre-tap-only channels first, split-N applies per tile); cblk_off[i] = output channel of 64-column block i.
  int nsplit, perm, cblk_off[8];
  uint32_t desc_hi_b, idesc_blk;
  // epilogue
  int cout, out_channels, out_coff, act, out_f32, is_bf16;
  void* out;
  const void* res0;
  const void* res1;
  int res0_channels, res1_channels;
  const float* bias;
  // skip computed in the epilogue (RM = 3): the skip tensor is a 1x1 conv (no activation) of the 8-channel network input
  // (6 channels + 2 zero pads), map_r is that input.  skip_w = [64][8] 16-bit: the folded weights of channels 0-5, and
  // the bias split in two 16-bit parts (hi, lo = bias - hi) in columns 6 and 7, which the kernel multiplies by 1
  int skip;
  const void* skip_w;
  // fused segmentation head (final conv only): softmax -> argmax -> mask; any of logits/probs may be NULL
  int head, none_index;
  const uint8_t* mask;
  float* probs;
  int32_t* preds;
  float* logits;
  unsigned long long* dbg;    // optional [gridDim.x][16] cycle counters (pcls_net_set_option "tc_debug")
};

// 16-bit pack of two floats with the ReLU fused into the conversion (cvt.rn.relu: exact - rounding is monotonic)
template <typename T> __device__ __forceinline__ uint32_t pack2_relu(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2_relu<__half>(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
template <> __device__ __forceinline__ uint32_t pack2_relu<__nv_bfloat16>(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

// packed 16-bit add (one instruction per two outputs)
template <typename T> __device__ __forceinline__ uint32_t add2_16(uint32_t a, uint32_t b);
template <> __device__ __forceinline__ uint32_t add2_16<__half>(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("add.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
template <> __device__ __forceinline__ uint32_t add2_16<__nv_bfloat16>(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}

// Skip computed in the epilogue (RM = 3): warp-level m16n8k8 MMAs (fp32 accumulation), the 16-bit results go through
// stmatrix into the output staging buffer, where the packed skip add reads them like a TMA-loaded residual block.
template <typename T> __device__ __forceinline__ uint32_t pack2_rn(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2_rn<__half>(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
template <> __device__ __forceinline__ uint32_t pack2_rn<__nv_bfloat16>(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
// d = a (16 x 8, row-major) * b (8 x 8, column-major), fp32 accumulators starting from zero
template <typename T> __device__ __forceinline__ void mma_16x8x8(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t b);
template <> __device__ __forceinline__ void mma_16x8x8<__half>(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t b) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%7, %7, %7, %7};"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]) : "r"(a0), "r"(a1), "r"(b), "f"(0.0f));
}
template <> __device__ __forceinline__ void mma_16x8x8<__nv_bfloat16>(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t b) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5}, {%6}, {%7, %7, %7, %7};"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]) : "r"(a0), "r"(a1), "r"(b), "f"(0.0f));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void stmatrix_x4(uint32_t addr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.shared.b16 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(r0), "r"(r1), "r"(r2), "r"(r3)
               : "memory");
}

// 8 accumulator columns (the bias is already in them: the epilogue pre-loads every TMEM accumulator with the bias row
// before its MMAs run, see preload_bias) -> activation, +residuals -> one 16-byte vector of 16-bit outputs.
// Without residuals ReLU rides in the float -> 16-bit conversion: 4 instructions per 8 outputs.  With residuals
// (added AFTER the activation, in float32): one max per element for ReLU / none (max(v, lo), lo = 0 / -inf), two for
// LeakyReLU(0.1).  LEAKY is a kernel template parameter: the epilogue's instruction count bounds the memory-side layers.
template <typename T, bool LEAKY, bool BIAS>
__device__ __forceinline__ int4 epilogue_vec8(const uint32_t* acc, const float* bias8, float lo, bool has_r0, const int4& r0,
                                              bool has_r1, const int4& r1) {
  if constexpr (!BIAS && !LEAKY) {
    if (!has_r0 && !has_r1) {
      int4 o;
      if (lo == 0.0f) {
        o.x = (int)pack2_relu<T>(__uint_as_float(acc[0]), __uint_as_float(acc[1]));
        o.y = (int)pack2_relu<T>(__uint_as_float(acc[2]), __uint_as_float(acc[3]));
        o.z = (int)pack2_relu<T>(__uint_as_float(acc[4]), __uint_as_float(acc[5]));
        o.w = (int)pack2_relu<T>(__uint_as_float(acc[6]), __uint_as_float(acc[7]));
      } else {
        const float f[8] = {__uint_as_float(acc[0]), __uint_as_float(acc[1]), __uint_as_float(acc[2]), __uint_as_float(acc[3]),
                            __uint_as_float(acc[4]), __uint_as_float(acc[5]), __uint_as_float(acc[6]), __uint_as_float(acc[7])};
        o = pack8<T>(f);
      }
      return o;
    }
  }
  if constexpr (!LEAKY) {
    // ReLU + ONE skip tensor (the FireDeconv expands of SqueezeSegV2: x = relu(bn(conv)) + skip): the activation value is
    // rounded to 16 bits by the converting ReLU and the skip is added with packed 16-bit adds - 8 + 4 + 4 instructions per
    // 8 outputs instead of 8 + 8 + 8 (unpack) + 8 + 4; one more 16-bit rounding than the float32 add.  ncu source view of
    // fire13's expand: the epilogue warps (two per scheduler) run a serial chain at ~7 cycles per instruction, 80 % of
    // their samples are wait / selected / short_sb / no_inst / branch_resolving - the instruction count IS the run time:
    // 0.284 -> 0.269 ms.  (Also tried: the bias through one extra K = 16 MMA per pixel block, ones x (hi, lo) bias tile -
    // correct, but 3 % slower: the accumulator's MMAs sit on the critical path of its epilogue group.)
    if (has_r0 && !has_r1 && lo == 0.0f) {
      float v[8];
      if constexpr (BIAS) {
        const float4 b0 = *reinterpret_cast<const float4*>(bias8);
        const float4 b1 = *reinterpret_cast<const float4*>(bias8 + 4);
        v[0] = __uint_as_float(acc[0]) + b0.x; v[1] = __uint_as_float(acc[1]) + b0.y; v[2] = __uint_as_float(acc[2]) + b0.z;
        v[3] = __uint_as_float(acc[3]) + b0.w; v[4] = __uint_as_float(acc[4]) + b1.x; v[5] = __uint_as_float(acc[5]) + b1.y;
        v[6] = __uint_as_float(acc[6]) + b1.z; v[7] = __uint_as_float(acc[7]) + b1.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[j]);
      }
      int4 o;
      o.x = (int)add2_16<T>(pack2_relu<T>(v[0], v[1]), (uint32_t)r0.x);
      o.y = (int)add2_16<T>(pack2_relu<T>(v[2], v[3]), (uint32_t)r0.y);
      o.z = (int)add2_16<T>(pack2_relu<T>(v[4], v[5]), (uint32_t)r0.z);
      o.w = (int)add2_16<T>(pack2_relu<T>(v[6], v[7]), (uint32_t)r0.w);
      return o;
    }
  }
  float v[8];
  if constexpr (BIAS) {   // (kernels with residuals: the bias is added here, not pre-loaded)
    const float4 b0 = *reinterpret_cast<const float4*>(bias8);
    const float4 b1 = *reinterpret_cast<const float4*>(bias8 + 4);
    v[0] = __uint_as_float(acc[0]) + b0.x; v[1] = __uint_as_float(acc[1]) + b0.y; v[2] = __uint_as_float(acc[2]) + b0.z;
    v[3] = __uint_as_float(acc[3]) + b0.w; v[4] = __uint_as_float(acc[4]) + b1.x; v[5] = __uint_as_float(acc[5]) + b1.y;
    v[6] = __uint_as_float(acc[6]) + b1.z; v[7] = __uint_as_float(acc[7]) + b1.w;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(acc[j]);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = LEAKY ? fmaxf(v[j], v[j] * 0.1f) : fmaxf(v[j], lo);
  if (has_r0) {
    float f[8];
    unpack8<T>(r0, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += f[j];
  }
  if (has_r1) {
    float f[8];
    unpack8<T>(r1, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += f[j];
  }
  return pack8<T>(v);
}

// RM = 1: the residual kernel specialised at compile time for ONE skip tensor that is TMA-loaded into the output staging
// buffers, TMA-store epilogue, ReLU or LeakyReLU (the FireDeconv expands of SqueezeSegV2, Darknet's enc1 / enc2 blocks).  The generic residual kernel carries the
// code of every residual mode (cp.async staging, per-chunk LDG, second residual) behind run-time flags that are tested per
// 8 outputs; the epilogue's instruction chain is what bounds these layers (DESIGN.md section 6, step 22).
template <typename T, int KC, int SUB, int G, bool RES, bool LEAKY, int KS = KC / 16, int RM = 0>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_r,
               const __grid_constant__ CUtensorMap map_b2, const __grid_constant__ CUtensorMap map_c2,
               const __grid_constant__ TcParams p, const int num_tiles) {
  constexpr bool PRELOAD = !RES;   // bias pre-loaded into the TMEM accumulators (see preload_bias)
  constexpr bool RTMA = RES && RM == 1;
  constexpr bool PTMA = !RES && RM == 2;   // no residual, 16-bit outputs through the TMA-store epilogue (known at compile time)
  // RM = 3: as RM = 1, but the skip is computed from the network input (TcParams::skip) instead of loaded, G = 4, ReLU
  constexpr bool SKIP = RES && RM == 3;
  static_assert(!SKIP || (G == 4 && !LEAKY), "the computed skip exists for the pixel-group view G = 4 with ReLU");
  constexpr bool FIXED = RTMA || SKIP;      // one skip tensor, TMA-store epilogue, known at compile time
  extern __shared__ uint8_t smem_raw[];
  // carve: [stages x (A tile | B tiles)] 1024-aligned, resident weights, barriers, TMEM base slot, bias
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int S = p.stages;
  const uint32_t a_bytes = (uint32_t)p.a_bytes, b_tile_bytes = (uint32_t)p.b_tile_bytes;
  const bool b_resident = p.b_resident != 0;
  const uint32_t b_stage_bytes = b_resident ? 0u : (uint32_t)SUB * b_tile_bytes;
  const uint32_t stage_bytes = a_bytes + b_stage_bytes;
  const uint32_t bres_base = smem_base + (uint32_t)S * stage_bytes;   // resident weights (1024-aligned)
  const uint32_t cstage_base = bres_base + (uint32_t)p.bres_bytes;  // output staging: [group][n_cbuf] x c_stage_bytes
  const uint32_t rstage_base = cstage_base + (p.tma_store ? (uint32_t)(p.n_cbuf * TC_NG) * (uint32_t)p.c_stage_bytes : 0u);  // residual0 staging (RES)
  // (SKIP: the same space holds two 8 KB network-input tiles per group)
  const uint32_t bar_base = rstage_base + ((RES && (SKIP || p.res_smem)) ? (uint32_t)TC_NG * 16384u : 0u);
#define FULL_BAR(s) (bar_base + 8u * (uint32_t)(s))
#define EMPTY_BAR(s) (bar_base + 8u * (uint32_t)(S + (s)))
#define TFULL_BAR(a) (bar_base + 8u * (uint32_t)(2 * S + (a)))
#define TEMPTY_BAR(a) (bar_base + 8u * (uint32_t)(2 * S + 8 + (a)))
#define BRES_BAR (bar_base + 8u * (uint32_t)(2 * S + 16))
#define RFULL_BAR(i) (bar_base + 8u * (uint32_t)(2 * S + 17 + (i)))   // [group][3]: residual block landed in staging buffer
                                                                       // (SKIP: [group][2] network-input tile landed)
  const uint32_t tmem_slot = bar_base + 8u * (uint32_t)(2 * S + 17 + 3 * TC_NG);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  float* bias_s = reinterpret_cast<float*>(smem_raw + (((tmem_slot + 16u + 15u) & ~15u) - smem_u32(smem_raw)));  // [n_nt * BN], 16-byte aligned
  for (int i = threadIdx.x; i < p.n_nt * p.BN; i += blockDim.x) bias_s[i] = p.bias[G > 1 ? i % p.cout_blk : i];
  float* head_s = bias_s + ((p.n_nt * p.BN + 3) & ~3);  // [4 * TC_NG warps][32][33] staging of the fused head (out_f32 layers)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // wait-cycle counters (tools/tc_debug_run.py): compiled in only with -DPCLS_TC_DEBUG=1, the `if (dbg)` tests and the
  // sixteen counter registers are measurable in the epilogue loops
  unsigned long long* const dbg = PCLS_TC_DEBUG ? p.dbg : nullptr;
  unsigned long long dbg_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const unsigned long long dbg_start = dbg ? clk() : 0ull;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    if (p.n1 > 0) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b2) : "memory");
    if (p.tma_store) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_c) : "memory");
    if (RES && (SKIP || p.res_tma)) asm volatile("prefetch.tensormap [%0];" ::"l"(&map_r) : "memory");
    for (int i = 0; i < 3 * TC_NG; ++i) mbar_init(RFULL_BAR(i), 1);
    for (int s = 0; s < S; ++s) { mbar_init(FULL_BAR(s), 1); mbar_init(EMPTY_BAR(s), 1); }
    for (int a = 0; a < 8; ++a) { mbar_init(TFULL_BAR(a), 1); mbar_init(TEMPTY_BAR(a), 4); }
    mbar_init(BRES_BAR, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {  // TMEM allocation: one warp, whole warp executes
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // PDL (common.cuh): the layer behind this one may start its prologue now; everything above (and the resident weight
  // loads of warp 0 below) is independent of the layer in front, all activation traffic comes after pdl_wait()
  pdl_trigger(p.pdl_early);
  if (warp != 0) pdl_wait();

  const int n_groups = p.n_groups, kchunks = p.kchunks, n_nt = p.n_nt, n_phase = p.n_phase, n_wt = p.n_wt, n_ht = p.n_ht;
  const int BN = p.BN;

  if (warp == 0) {
    // ===================== TMA producer (whole warp, one elected lane issues) =====================
    {
      if (b_resident) {
        // weight-stationary: every weight tile of the layer once per CTA, laid out in MMA iteration order
        // [phase][group][K chunk][sub] so that the issuer only increments an address
        mbar_arrive_expect_tx_elect(BRES_BAR, (uint32_t)p.bres_tx);
        uint32_t dst = bres_base;
        const int n0r = p.nsplit ? (int)(blockIdx.x % (unsigned)n_nt) * BN : 0;   // this CTA's N tile (N-split across CTAs)
        for (int ph = 0; ph < n_phase; ++ph)
          for (int g = 0; g < n_groups; ++g)
            for (int kc = 0; kc < kchunks; ++kc)
#pragma unroll
              for (int u = 0; u < SUB; ++u) {
                const int tap = p.grp_w[ph][g][u];
                if (p.n1 > 0 && tap != 4) {   // rows [n1, BN) only
                  tma_load_3d_elect(dst, &map_b2, BRES_BAR, kc * KC, n0r + p.n1, tap);
                  dst += (uint32_t)p.b_small_bytes;
                } else {
                  tma_load_3d_elect(dst, &map_b, BRES_BAR, kc * KC, n0r, tap);
                  dst += b_tile_bytes;
                }
              }
      }
      pdl_wait();   // weights are in flight; the activations need the producing layer to have finished
      const uint32_t a_tx_bytes = (uint32_t)(p.a_rows * KC * 2);
      const int BW = p.BW, BH = p.BH;
      const bool is5d = p.a_is_5d != 0;
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int r = tile;
        const int nt = r % n_nt; r /= n_nt;
        const int ph = r % n_phase; r /= n_phase;
        const int wt = r % n_wt; r /= n_wt;
        const int ht = r % n_ht;
        const int b = r / n_ht;
        const int w0 = wt * BW, h0 = ht * BH, n0 = nt * BN;
        for (int g = 0; g < n_groups; ++g) {
          const int hh = h0 + p.grp_dh[ph][g], ww = w0 + p.grp_dw[ph][g], par = p.grp_par[ph][g];
          int wtap[SUB];
#pragma unroll
          for (int u = 0; u < SUB; ++u) wtap[u] = p.grp_w[ph][g][u];
          for (int kc = 0; kc < kchunks; ++kc) {
            { DBG_T0; mbar_wait(EMPTY_BAR(stage), phase ^ 1u); DBG_ADD(0); }
            const uint32_t a_dst = smem_base + (uint32_t)stage * stage_bytes;
            const uint32_t fb = FULL_BAR(stage);
            uint32_t tx_bytes = a_tx_bytes;
            if (!b_resident) {
#pragma unroll
              for (int u = 0; u < SUB; ++u) tx_bytes += (p.n1 > 0 && wtap[u] != 4) ? (uint32_t)p.b_small_bytes : b_tile_bytes;
            }
            mbar_arrive_expect_tx_elect(fb, tx_bytes);
            if (is5d) tma_load_5d_elect(a_dst, &map_a, fb, kc * KC, par, ww, hh, b);
            else tma_load_4d_elect(a_dst, &map_a, fb, kc * KC, ww, hh, b);
            if (!b_resident) {
#pragma unroll
              for (int u = 0; u < SUB; ++u) {
                if (p.n1 > 0 && wtap[u] != 4)
                  tma_load_3d_elect(a_dst + a_bytes + (uint32_t)u * b_tile_bytes, &map_b2, fb, kc * KC, p.n1, wtap[u]);
                else
                  tma_load_3d_elect(a_dst + a_bytes + (uint32_t)u * b_tile_bytes, &map_b, fb, kc * KC, n0, wtap[u]);
              }
            }
            if (++stage == S) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp, one elected lane issues) =====================
    {
      const uint32_t desc_hi = p.desc_hi, idesc = p.idesc;
      const uint32_t n_acc = (uint32_t)p.n_acc;
      uint32_t sub_off[SUB];
#pragma unroll
      for (int u = 0; u < SUB; ++u) sub_off[u] = (uint32_t)(p.sub_row[u] * KC * 2);
      const int k_iters = n_groups * kchunks;
      const uint32_t bres_phase_bytes = (uint32_t)(k_iters * SUB) * b_tile_bytes;
      int stage = 0;
      uint32_t phase = 0, acc = 0, acc_phase = 0;
      if (b_resident) mbar_wait(BRES_BAR, 0u);
      const int my_tiles = (num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
      for (int seq = 0; seq < my_tiles; ++seq) {
        const int tile = blockIdx.x + seq * gridDim.x;   // (only the transposed-conv phase below reads it)
        { DBG_T0; mbar_wait(TEMPTY_BAR(acc), PRELOAD ? acc_phase : (acc_phase ^ 1u)); DBG_ADD(1); }  // the epilogue has drained this accumulator and pre-loaded the bias row
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * (uint32_t)BN;
        uint32_t b_res = bres_base + (n_phase > 1 ? (uint32_t)((tile / n_nt) % n_phase) * bres_phase_bytes : 0u);
        uint32_t accumulate = PRELOAD ? 1u : 0u, acc_lo = accumulate;   // PRELOAD: the accumulator starts from the bias row
        int kc_i = 0, g_i = 0;   // K chunk and A-load group of iteration k
        for (int k = 0; k < k_iters; ++k) {
          { DBG_T0; mbar_wait(FULL_BAR(stage), phase); DBG_ADD(2); }
          const uint32_t a_addr = smem_base + (uint32_t)stage * stage_bytes;
          tc_fence_after();
          if constexpr (G == 1) {
            uint32_t b_addr = b_resident ? b_res : a_addr + a_bytes;
            const uint32_t n1 = (uint32_t)p.n1;
#pragma unroll
            for (int u = 0; u < SUB; ++u) {
              // descriptors: start address (>>4) | LBO = 1 in the low word; SBO / version / swizzle mode in the high word.
              // A row-shifted start (halo taps) needs no base offset: the swizzle is a function of absolute smem address bits.
              const uint64_t a_desc = ((uint64_t)desc_hi << 32) | (uint64_t)((((a_addr + sub_off[u]) >> 4) & 0x3FFFu) | 0x10000u);
              const uint64_t b_desc = ((uint64_t)desc_hi << 32) | (uint64_t)(((b_addr >> 4) & 0x3FFFu) | 0x10000u);
              if (n1 == 0u) {
#pragma unroll
                for (int j = 0; j < KS; ++j) {  // +32 bytes along K inside the swizzle atom per UMMA_K = 16
                  umma_f16_elect(d_tmem, a_desc + (uint64_t)(2 * j), b_desc + (uint64_t)(2 * j), idesc, accumulate);
                  accumulate = 1u;
                }
                b_addr += b_tile_bytes;
              } else if (p.grp_w[0][g_i][u] != 4) {
                // split-N, outer tap: the tile holds weight rows [n1, BN) only -> accumulator columns [n1, BN)
#pragma unroll
                for (int j = 0; j < KC / 16; ++j) {
                  umma_f16_elect(d_tmem + n1, a_desc + (uint64_t)(2 * j), b_desc + (uint64_t)(2 * j), p.idesc_small, accumulate);
                  accumulate = 1u;
                }
                b_addr += b_resident ? (uint32_t)p.b_small_bytes : b_tile_bytes;
              } else {
                // split-N, centre tap: full tile; columns [0, n1) see only this tap, columns [n1, BN) continue to accumulate
                const uint32_t b_hi = b_addr + n1 * (uint32_t)(KC * 2);
                const uint64_t b_desc_hi = ((uint64_t)desc_hi << 32) | (uint64_t)(((b_hi >> 4) & 0x3FFFu) | 0x10000u);
#pragma unroll
                for (int j = 0; j < KC / 16; ++j) {
                  umma_f16_elect(d_tmem, a_desc + (uint64_t)(2 * j), b_desc + (uint64_t)(2 * j), p.idesc_lo, acc_lo);
                  umma_f16_elect(d_tmem + n1, a_desc + (uint64_t)(2 * j), b_desc_hi + (uint64_t)(2 * j), p.idesc_small, accumulate);
                  acc_lo = 1u; accumulate = 1u;
                }
                b_addr += b_tile_bytes;
              }
            }
            if (b_resident) b_res = b_addr;
          } else {
            // pixel-group view, banded issue: output pixel p of the group and horizontal tap u read input pixel
            // t = p + u - 1, i.e. group dq = floor(t / G) (row offset dq + 1 in the halo tile) and K offset (t mod G) * Cin;
            // the product lands in accumulator columns [p * cout_blk, ..).  One small MMA per (p, u, 16 channels).
            constexpr int CIN = KC / G;
            const uint32_t desc_hi_b = p.desc_hi_b, idesc_blk = p.idesc_blk, cout_blk = (uint32_t)p.cout_blk;
#pragma unroll
            for (int u = 0; u < SUB; ++u) {
              const uint32_t b_addr = b_res + (uint32_t)u * b_tile_bytes;
              const uint64_t b_desc = ((uint64_t)desc_hi_b << 32) | (uint64_t)(((b_addr >> 4) & 0x3FFFu) | 0x10000u);
#pragma unroll
              for (int pp = 0; pp < G; ++pp) {
                constexpr int dummy = 0; (void)dummy;
                const int t = pp + (SUB == 3 ? u - 1 : 0);
                const int dq = t < 0 ? -1 : (t >= G ? 1 : 0);
                const int par = t - dq * G;
                const uint32_t a_start = a_addr + (uint32_t)((SUB == 3 ? dq + 1 : 0) * KC * 2 + par * CIN * 2);
                const uint64_t a_desc = ((uint64_t)desc_hi << 32) | (uint64_t)(((a_start >> 4) & 0x3FFFu) | 0x10000u);
#pragma unroll
                for (int j = 0; j < CIN / 16; ++j)
                  umma_f16_elect(d_tmem + (uint32_t)pp * cout_blk, a_desc + (uint64_t)(2 * j), b_desc + (uint64_t)(2 * j),
                           idesc_blk, (PRELOAD || (k | u | j) != 0) ? 1u : 0u);
              }
            }
          }
          if constexpr (G > 1) b_res += (uint32_t)SUB * b_tile_bytes;
          if (++kc_i == kchunks) { kc_i = 0; ++g_i; }
          umma_commit_elect(EMPTY_BAR(stage));  // smem slot free once these MMAs have read it
          if (++stage == S) { stage = 0; phase ^= 1u; }
        }
        umma_commit_elect(TFULL_BAR(acc));  // accumulator complete
        if (++acc == n_acc) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===================== epilogue: two warp-groups, alternate tiles =====================
    const int grp = (warp - 2) >> 2;
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int m = q * 32 + lane;
    const int ml_h = m >> p.bw_shift, ml_w = m & (p.BW - 1);
    const uint32_t n_acc = (uint32_t)p.n_acc;
    const int BW = p.BW, BH = p.BH, Hgrid = p.Hgrid, Wgrid = p.Wgrid, Wout = p.Wout, out_wmul = p.out_wmul;
    const int cout = p.cout, out_channels = p.out_channels, out_coff = p.out_coff;
    const int blk_shift = p.cout_blk_shift;              // pixel-group view: column n -> pixel n >> blk_shift
    const int blk_mask = G > 1 ? (1 << blk_shift) - 1 : -1;
    const float slope = p.act == PCLS_ACT_RELU ? 0.0f : (p.act == PCLS_ACT_LEAKY ? 0.1f : 1.0f);   // (float32 logits path)
    const float act_lo = (FIXED || p.act == PCLS_ACT_RELU) ? 0.0f : -INFINITY;
    const uint16_t* res0 = reinterpret_cast<const uint16_t*>(p.res0);
    const uint16_t* res1 = reinterpret_cast<const uint16_t*>(p.res1);
    const int res0_channels = p.res0_channels, res1_channels = p.res1_channels;
    const bool has_r0 = FIXED || res0 != nullptr, has_r1 = !FIXED && res1 != nullptr;
    const bool tma_store = FIXED || PTMA || p.tma_store != 0, out_f32 = !FIXED && !PTMA && p.out_f32 != 0, c_is_5d = p.c_is_5d != 0;
    const uint32_t c_stage_bytes = (uint32_t)p.c_stage_bytes;
    T* const outp = reinterpret_cast<T*>(p.out);
    const bool issuer = (q == 2) && lane == 0;            // first warp of the group (warp 2 or 6) issues the TMA stores
    const int bar_id = 1 + grp;
    // a group may only ever wait on the CURRENT or NEXT phase of an accumulator barrier (parity waits alias beyond that):
    // never run more groups than there are accumulators
    const uint32_t ng = n_acc < (uint32_t)TC_NG ? n_acc : (uint32_t)TC_NG;
    uint32_t tl = 0, blk = 0;
    const uint32_t nrb = (uint32_t)p.n_cbuf;   // staging buffers per group (res_tma: 3, or 2 when smem is short)
    // res_tma: TMA load of the residual block (tile, channel block cb) into staging buffer `bi` of this group
    auto issue_res = [&](int rtile, int rcb, uint32_t bi) {
      int r2 = rtile;
      const int nt2 = r2 % n_nt; r2 /= n_nt;
      const int ph2 = r2 % n_phase; r2 /= n_phase;
      const int wt2 = r2 % n_wt; r2 /= n_wt;
      const int ht2 = r2 % n_ht;
      const int b2 = r2 / n_ht;
      const uint32_t dst = cstage_base + (uint32_t)(grp * p.n_cbuf + (int)bi) * c_stage_bytes;
      const uint32_t bar = RFULL_BAR(grp * 3 + (int)bi);
      const int pp2 = G > 1 ? (nt2 * BN + rcb) >> blk_shift : 0;
      const int c02 = out_coff + (p.perm ? p.cblk_off[(nt2 * BN + rcb) >> 6] : ((nt2 * BN + rcb) & blk_mask));
      mbar_arrive_expect_tx(bar, 128u * 64u * 2u);
      if (c_is_5d) tma_load_5d(dst, &map_r, bar, c02, G > 1 ? pp2 : ph2, wt2 * BW, ht2 * BH, b2);
      else tma_load_4d(dst, &map_r, bar, c02, wt2 * BW, ht2 * BH, b2);
    };
    // the CTA's seq-th tile as a flat index of the (nt, phase, wt, ht, b) encoding, or -1 past the end
    auto tile_at = [&](uint32_t seq) -> int {
      const long long t = (long long)blockIdx.x + (long long)seq * gridDim.x;
      return t < num_tiles ? (int)t : -1;
    };
    if (RES && !SKIP && p.res_tma != 0 && has_r0 && issuer && (uint32_t)grp < ng && tile_at((uint32_t)grp) >= 0)
      issue_res(tile_at((uint32_t)grp), 0, 0u);
    // ---- SKIP: skip = 1x1 conv (6 -> 64, folded BN, no activation) of the 8-channel network input, computed here ----
    // A tile is 512 consecutive pixels of one image row, i.e. 8 KB of the input: ONE TMA load of 128 rows x 64 bytes (four
    // pixels per row, SWIZZLE_64B) per tile, a tile ahead, into one of two buffers per group.  For the 64-channel block of
    // pixel pp the warp's 32 rows m take pixel 4m + pp: two 16-row MMA tiles x eight 8-channel N tiles of m16n8k8, A by
    // ldmatrix (the 64-byte swizzle puts the 8 rows of a matrix in distinct banks), B = the weights in registers, C = the
    // bias; the results are rounded to 16 bits and written by stmatrix into the swizzled staging rows that the packed
    // skip add reads.  Each warp reads back only its own 32 rows.
    uint32_t skw[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint32_t in_base = rstage_base + (uint32_t)grp * 16384u;   // [2] x 8 KB
    // the bias rides in the MMA: lanes holding input channels 6 and 7 (the zero pads) put 1 there instead
    const bool ones_lane = (lane & 3) == 3;
    const uint32_t one2 = std::is_same<T, __half>::value ? 0x3C003C00u : 0x3F803F80u;
    if constexpr (SKIP) {
      const uint32_t* w32 = reinterpret_cast<const uint32_t*>(p.skip_w);   // [64][8] 16-bit: row n, channels 2 t, 2 t + 1
#pragma unroll
      for (int j = 0; j < 8; ++j) skw[j] = __ldg(w32 + (8 * j + (lane >> 2)) * 4 + (lane & 3));
    }
    auto issue_in = [&](int rtile, uint32_t bi) {
      const int wt2 = (rtile / n_nt / n_phase) % n_wt;
      const int ht2 = (rtile / n_nt / n_phase / n_wt) % n_ht;
      const int b2 = rtile / n_nt / n_phase / n_wt / n_ht;
      const uint32_t bar = RFULL_BAR(grp * 3 + (int)bi);
      mbar_arrive_expect_tx(bar, 8192u);
      tma_load_4d(in_base + bi * 8192u, &map_r, bar, 0, wt2 * BW, ht2 * BH, b2);
    };
    auto compute_skip = [&](uint32_t buf, int pp, uint32_t in_buf) {
      uint32_t a[4];
      ldmatrix_x4(in_buf + (uint32_t)(m * 64) + (uint32_t)((pp ^ ((m >> 1) & 3)) << 4), a);
#pragma unroll
      for (int k = 0; k < 4; ++k) a[k] = ones_lane ? one2 : a[k];
      const int sr = (q * 32 + ((lane >> 3) & 1) * 8 + (lane & 7));   // stmatrix row of this lane (M tile 0)
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int jp = 0; jp < 4; ++jp) {
          float d0[4], d1[4];
          mma_16x8x8<T>(d0, a[2 * i], a[2 * i + 1], skw[2 * jp]);
          mma_16x8x8<T>(d1, a[2 * i], a[2 * i + 1], skw[2 * jp + 1]);
          const uint32_t chunk = (uint32_t)((2 * jp + (lane >> 4)) ^ (lane & 7));
          stmatrix_x4(buf + (uint32_t)((sr + 16 * i) * 128) + (chunk << 4), pack2_rn<T>(d0[0], d0[1]), pack2_rn<T>(d0[2], d0[3]),
                      pack2_rn<T>(d1[0], d1[1]), pack2_rn<T>(d1[2], d1[3]));
        }
      __syncwarp();
    };
    if (SKIP && issuer && (uint32_t)grp < ng && tile_at((uint32_t)grp) >= 0) issue_in(tile_at((uint32_t)grp), 0u);
    // Bias through the accumulator (kernels without residuals): before an accumulator's MMAs start, its rows are pre-loaded with the bias row of
    // the tile that will use it (tcgen05.st, 4x the TMEM read rate; every MMA then accumulates).  This takes the bias
    // add - one FADD per output element plus the shared-memory reads of the bias - out of the epilogue's inner loop.
    // Done by the group that owns the accumulator: once up front, then right after draining it, for the tile n_acc later.
    // (Measured: the residual kernels - epilogue-bound, 166 registers - lose 9 % with it, interleaved with the chunk reads
    // or not; they keep the bias add in the epilogue.)
    auto preload_bias = [&](uint32_t a, int tile_next) {
      if (tile_next >= 0) {
        const float* bsrc = bias_s + (tile_next % n_nt) * BN;
        const uint32_t t_dst = tmem_base + ((uint32_t)(q * 32) << 16) + a * (uint32_t)BN;
#pragma unroll 1
        for (int c = 0; c + 32 <= BN; c += 32) {
          uint32_t bv[32];
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 t4 = *reinterpret_cast<const float4*>(bsrc + c + j);
            bv[j] = __float_as_uint(t4.x); bv[j + 1] = __float_as_uint(t4.y); bv[j + 2] = __float_as_uint(t4.z); bv[j + 3] = __float_as_uint(t4.w);
          }
          tmem_st32(t_dst + (uint32_t)c, bv);
        }
        if (BN & 16) {
          uint32_t bv[16];
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 t4 = *reinterpret_cast<const float4*>(bsrc + (BN & ~31) + j);
            bv[j] = __float_as_uint(t4.x); bv[j + 1] = __float_as_uint(t4.y); bv[j + 2] = __float_as_uint(t4.z); bv[j + 3] = __float_as_uint(t4.w);
          }
          tmem_st16(t_dst + (uint32_t)(BN & ~31), bv);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(TEMPTY_BAR(a));
    };
    if (PRELOAD && (uint32_t)grp < ng)
      for (uint32_t a = (uint32_t)grp; a < n_acc; a += ng) preload_bias(a, tile_at(a));
    for (; (uint32_t)grp < ng; ++tl) {
      const int tile = tile_at(tl);
      if (tile < 0) break;
      if ((int)(tl % ng) != grp) continue;
      int r = tile;
      const int nt = r % n_nt; r /= n_nt;
      const int ph = r % n_phase; r /= n_phase;
      const int wt = r % n_wt; r /= n_wt;
      const int ht = r % n_ht;
      const int b = r / n_ht;
      const int h = ht * BH + ml_h, w = wt * BW + ml_w;
      const bool valid = h < Hgrid && w < Wgrid;
      const int64_t pix = ((int64_t)b * Hgrid + h) * Wout + (int64_t)w * out_wmul + ph;
      const uint32_t acc = tl & (n_acc - 1u), acc_parity = (tl / n_acc) & 1u;
      const int n0 = nt * BN;
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + acc * (uint32_t)BN;
      // element offset of (this row's pixel-in-group, channel) for accumulator column n, or -1 when out of range
      auto elem_off = [&](int n, int channels) -> int64_t {
        const int pp = G > 1 ? n >> blk_shift : 0;
        const int co = n & blk_mask;
        return (valid && co + 8 <= cout) ? (pix + pp) * channels + out_coff + co : (int64_t)-1;
      };
      // Residual rows (RES kernels only).  residual0 of a 128-column batch is copied global -> shared with cp.async
      // (16 bytes per vector, thread-private slots, zero-fill for out-of-range rows) BEFORE waiting for the accumulator:
      // no registers are held, the DRAM latency overlaps the MMAs of this tile and the chunk loop stays compact.
      // The second residual (Darknet decoder only, compute-bound layers) is fetched one chunk ahead.
      const uint32_t rslot = rstage_base + (uint32_t)grp * 16384u + (uint32_t)(m & 127) * 16u;  // + i * 2048 per vector
      int4 r0[4], r1[4];
      const bool res_smem = !FIXED && RES && p.res_smem != 0 && has_r0;
      const bool res_tma = RTMA || (RES && !SKIP && p.res_tma != 0 && has_r0);
      const bool res_stage = res_tma || SKIP;   // residual0 block sits in the output staging buffer (row res_row)
      uint32_t res_row = 0;     // res_tma: this thread's row of the staging buffer that holds the residual block
      auto prefetch_r0 = [&](int cs) {
        if constexpr (RES) {
          if (res_smem) {
#pragma unroll 4
            for (int i = 0; i < 8; ++i) {
              const int64_t o = (cs + i * 8 < BN) ? elem_off(n0 + cs + i * 8, res0_channels) : (int64_t)-1;
              cp_async16(rslot + (uint32_t)i * 2048u, res0 + (o >= 0 ? o : 0), o >= 0);
            }
            cp_async_commit();
          }
        }
      };
      auto load_r1 = [&](int c) {   // register path: residual1, and residual0 when it is not staged through smem
        if constexpr (RES) {
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const int64_t o = has_r1 ? elem_off(n0 + c + g * 8, res1_channels) : (int64_t)-1;
            r1[g] = o >= 0 ? __ldg(reinterpret_cast<const int4*>(res1 + o)) : make_int4(0, 0, 0, 0);
            if (has_r0 && !res_smem && !res_stage) {
              const int64_t o0 = elem_off(n0 + c + g * 8, res0_channels);
              r0[g] = o0 >= 0 ? __ldg(reinterpret_cast<const int4*>(res0 + o0)) : make_int4(0, 0, 0, 0);
            }
          }
        }
      };
      const bool reg_res = RES && (has_r1 || (has_r0 && !res_smem && !res_stage));
      prefetch_r0(0);
      if (reg_res) load_r1(0);
      uint8_t head_mask = 1;                                       // fused head: the mask byte travels during the MMAs
      if (out_f32 && p.head && valid) head_mask = p.mask[pix];
      { DBG_T0; mbar_wait(TFULL_BAR(acc), acc_parity); DBG_ADD(3); }
      const unsigned long long _te = dbg ? clk() : 0ull;
      tc_fence_after();
      if (res_smem) cp_async_wait_all();
      // one 32-column chunk of accumulator registers -> 4 output vectors, handed to `sink(g, vector)`
      auto process = [&](const uint32_t* v, int cc, auto&& sink) {
        if constexpr (RES) {
          if (res_smem && cc > 0 && (cc & 63) == 0) { prefetch_r0(cc); cp_async_wait_all(); }  // next 64-column batch
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          int4 r0v = make_int4(0, 0, 0, 0);
          if constexpr (RES) {
            r0v = res_stage ? ld_shared_v4(res_row + (uint32_t)(((((cc & 63) >> 3) + g) ^ (m & 7)) << 4))
                : res_smem ? ld_shared_v4(rslot + (uint32_t)(((cc & 63) >> 3) + g) * 2048u) : r0[g];
          }
          sink(g, epilogue_vec8<T, LEAKY, !PRELOAD>(v + g * 8, bias_s + n0 + cc + g * 8, act_lo, RES && has_r0, r0v, RES && has_r1, r1[g]));
        }
        if (reg_res && cc + 32 < BN) load_r1(cc + 32);
      };
      // TMEM -> registers -> process, one chunk at a time (direct-store path)
      auto chunk = [&](int cc, auto&& sink) {
        uint32_t v[32];
        if (cc + 32 <= BN) {
          tmem_ld32(t_row + (uint32_t)cc, v);
        } else {  // BN % 32 == 16 tail
          uint32_t v16[16];
          tmem_ld16(t_row + (uint32_t)cc, v16);
#pragma unroll
          for (int j = 0; j < 16; ++j) { v[j] = v16[j]; v[16 + j] = 0u; }
        }
        tmem_ld_wait();
        process(v, cc, sink);
      };
      // hands the accumulator back to the MMA issuer (PRELOAD: after writing the next tile's bias row into it)
      bool released = false;
      auto release_acc = [&]() {
        released = true;
        if constexpr (PRELOAD) {
          preload_bias(acc, tile_at(tl + n_acc));
        } else {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(TEMPTY_BAR(acc));
        }
      };
      if (out_f32) {
        // float32 logits (conv14 / head layer), cout <= 32.  With the fused head the softmax / argmax / mask of
        // nets/SegmentationNetwork.py:58-69 run here on the accumulator registers: logits never travel to HBM unless
        // the caller asks for them.  Each warp stages 32 pixels x cout floats in smem so that global stores are coalesced.
        float lg[32];
        {
          uint32_t v[32];
          if (BN >= 32) {
            tmem_ld32(t_row, v);
          } else {
            uint32_t v16[16];
            tmem_ld16(t_row, v16);
#pragma unroll
            for (int j = 0; j < 16; ++j) { v[j] = v16[j]; v[16 + j] = 0u; }
          }
          tmem_ld_wait();
          // columns >= cout (padding up to the next multiple of 4) become -inf: the loops below run in uniform blocks
          // of four classes without per-class range checks
#pragma unroll
          for (int c4 = 0; c4 < 32; c4 += 4) {
            if (c4 < cout) {
#pragma unroll
              for (int j = c4; j < c4 + 4; ++j) {
                const float x = __uint_as_float(v[j]) + (PRELOAD ? 0.0f : bias_s[n0 + j]);   // (PRELOAD: the bias is in the accumulator)
                lg[j] = (j < cout) ? fmaxf(x, x * slope) : -INFINITY;
              }
            }
          }
        }
        float* stg = head_s + (warp - 2) * (32 * 33);
        const int64_t pix0 = __shfl_sync(0xffffffffu, pix, 0);      // pixels of a warp are consecutive in memory
        const int n_valid = __popc(__ballot_sync(0xffffffffu, valid));
        auto write_rows = [&](float* dst) {                          // lg[] of 32 pixels -> dst[pix0*cout ..] coalesced
          if ((cout & 3) == 0) {
            // the warp's rows form ONE contiguous span of the output: stage them in that layout, one bulk copy
            if (lane == 0) bulk_wait_read0();                        // the previous copy has finished reading the rows
            __syncwarp();
#pragma unroll
            for (int c4 = 0; c4 < 32; c4 += 4)
              if (c4 < cout) *reinterpret_cast<float4*>(stg + lane * cout + c4) = make_float4(lg[c4], lg[c4 + 1], lg[c4 + 2], lg[c4 + 3]);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0 && n_valid > 0) {
              bulk_store_1d(dst + pix0 * cout, smem_u32(stg), (uint32_t)(n_valid * cout * 4));
              bulk_commit();
            }
            return;
          }
          __syncwarp();
#pragma unroll
          for (int c = 0; c < 32; ++c) if (c < cout) stg[lane * 33 + c] = lg[c];
          __syncwarp();
          const int n_el = n_valid * cout;
          int px = lane / cout, cc = lane - px * cout;               // (pixel, class) of element `lane`, advanced by 32
          const int dpx = 32 / cout, dcc = 32 - dpx * cout;
          for (int e = lane; e < n_el; e += 32) {
            dst[pix0 * cout + e] = stg[px * 33 + cc];
            px += dpx; cc += dcc;
            if (cc >= cout) { cc -= cout; ++px; }
          }
        };
        if (!p.head) {
          if (valid) {
            float* o = reinterpret_cast<float*>(p.out) + pix * out_channels + out_coff;
#pragma unroll
            for (int c = 0; c < 32; ++c) if (c < cout) o[c] = lg[c];
          }
        } else {
          if (p.logits) write_rows(p.logits);
          // softmax with SFU exponentials and one reciprocal (<= 2 ulp from the standalone head's expf / IEEE division),
          // argmax over the rounded probabilities, first index on ties
          float mx = lg[0];
#pragma unroll
          for (int c4 = 0; c4 < 32; c4 += 4)
            if (c4 < cout) mx = fmaxf(fmaxf(mx, fmaxf(lg[c4], lg[c4 + 1])), fmaxf(lg[c4 + 2], lg[c4 + 3]));
          float sum = 0.0f;
#pragma unroll
          for (int c4 = 0; c4 < 32; c4 += 4)
            if (c4 < cout) {
#pragma unroll
              for (int j = c4; j < c4 + 4; ++j) { lg[j] = ex2_ftz((lg[j] - mx) * 1.4426950408889634f); sum += lg[j]; }
            }
          const float inv = __fdividef(1.0f, sum);
          int best = 0;
          float bp = -1.0f;
#pragma unroll
          for (int c4 = 0; c4 < 32; c4 += 4)
            if (c4 < cout) {
#pragma unroll
              for (int j = c4; j < c4 + 4; ++j) { lg[j] *= inv; if (lg[j] > bp) { bp = lg[j]; best = j; } }
            }
          if (valid) {
            if (head_mask == 0) best = p.none_index;
            p.preds[pix] = best;
          }
          if (p.probs) write_rows(p.probs);
        }
      } else if (tma_store) {
        // ---- TMEM -> registers -> swizzled smem tile -> TMA bulk tensor store (full lines, edges clipped by TMA) ----
        // blocks of 64 channels (128-byte rows, SWIZZLE_128B).  The accumulator reads are double-buffered: the tcgen05.ld
        // of chunk c + 1 is in flight while chunk c is processed, and the accumulator goes back to the MMA issuer as soon
        // as its LAST chunk sits in registers - one chunk of processing (1/8 of the drain of a 256-column tile) earlier,
        // which covers the ~2000 cycles the next tile's MMAs take (n_acc = 2 with two groups: each group waits for ITS
        // accumulator, so that latency sat on the group's critical path: wait-tfull was 10-12 % of fire11-13's expands).
        // (Not for the residual kernels of the plain view - fire10's N-split expand, Darknet's blocks: 168 registers are
        // the cap, the second buffer spills there: fire10 0.170 -> 0.186 ms.)
        constexpr bool DBUF = !(RES && G == 1);
        uint32_t va[32], vb[DBUF ? 32 : 1];
        if constexpr (DBUF) tmem_ld32(t_row, va);
        for (int cb = 0; cb < BN; cb += 64, ++blk) {
          uint32_t buf;
          if (res_tma) {
            // three staging buffers per group.  Block k+1's residual is TMA-loaded into buffer (k+1) % 3 while block k is
            // computed: the buffer is free once the store of block k-2 has read it (stores k-2 .. k-1 may be pending).
            if (issuer) {
              int ntile = tile, ncb = cb + 64;
              if (ncb >= BN) { ncb = 0; ntile = tile_at(tl + ng); }
              if (ntile >= 0) {
                // three buffers: store k-1 may still be reading its buffer; two buffers: it must have finished (same buffer)
                if (nrb == 3u) bulk_wait_read1(); else bulk_wait_read0();
                issue_res(ntile, ncb, (blk + 1u) % nrb);
              }
            }
            buf = cstage_base + (uint32_t)(grp * (int)nrb + (int)(blk % nrb)) * c_stage_bytes;
            { DBG_T0; mbar_wait(RFULL_BAR(grp * 3 + (int)(blk % nrb)), (blk / nrb) & 1u); DBG_ADD(4); }
          } else {
            // two staging buffers per group: block k is written while the TMA store of block k-1 drains the other one
            buf = cstage_base + (uint32_t)(grp * 2 + (int)(blk & 1u)) * c_stage_bytes;
            if constexpr (SKIP) {
              const uint32_t tg = tl / ng;   // this group's tile count: input buffer tg & 1
              if (cb == 0) {
                // the other input buffer was last read by the previous tile, before its last group barrier
                if (issuer && tile_at(tl + ng) >= 0) issue_in(tile_at(tl + ng), (tg + 1u) & 1u);
                DBG_T0; mbar_wait(RFULL_BAR(grp * 3 + (int)(tg & 1u)), (tg >> 1) & 1u); DBG_ADD(4);
              }
              // buffer blk & 1 was last read by the store of block k-2, finished before block k-1's group barrier
              compute_skip(buf, cb >> 6, in_base + (tg & 1u) * 8192u);
            }
          }
          // a 32-channel tail block (N tile = 64 k + 32, kernels without residuals): 64-byte rows, SWIZZLE_64B, map_c2
          const bool narrow = !RES && BN - cb < 64;
          const uint32_t row_addr = buf + (uint32_t)(m * (narrow ? 64 : 128));
          res_row = row_addr;
          if constexpr (!DBUF) {
#pragma unroll 1
            for (int ci = 0; ci < 2; ++ci)
              chunk(cb + ci * 32, [&](int g, const int4& o) {
                st_shared_v4(row_addr + (uint32_t)(((ci * 4 + g) ^ (m & 7)) << 4), o); });
          } else if (narrow) {   // (always the last block of the tile)
            tmem_ld_wait();
            release_acc();
            process(va, cb, [&](int g, const int4& o) { st_shared_v4(row_addr + (uint32_t)((g ^ ((m >> 1) & 3)) << 4), o); });
          } else {
            tmem_ld_wait();
            tmem_ld32(t_row + (uint32_t)(cb + 32), vb);
            process(va, cb, [&](int g, const int4& o) { st_shared_v4(row_addr + (uint32_t)((g ^ (m & 7)) << 4), o); });
            tmem_ld_wait();
            if (cb + 64 < BN) tmem_ld32(t_row + (uint32_t)(cb + 64), va);
            else release_acc();
            process(vb, cb + 32, [&](int g, const int4& o) { st_shared_v4(row_addr + (uint32_t)(((4 + g) ^ (m & 7)) << 4), o); });
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // smem writes -> visible to the TMA engine
          if (!res_tma) { DBG_T0; if (issuer) bulk_wait_read0(); DBG_ADD(4); }   // store k-1 has finished reading the OTHER buffer
          { DBG_T0; group_barrier(bar_id); DBG_ADD(5); }
          if (issuer) {
            const int pp = G > 1 ? (n0 + cb) >> blk_shift : 0;
            const int c0 = out_coff + (p.perm ? p.cblk_off[(n0 + cb) >> 6] : ((n0 + cb) & blk_mask));
            if (c_is_5d) tma_store_5d(&map_c, buf, c0, G > 1 ? pp : ph, wt * BW, ht * BH, b);
            else tma_store_4d(narrow ? &map_c2 : &map_c, buf, c0, wt * BW, ht * BH, b);
            bulk_commit();
          }
        }
      } else {
        // ---- direct 16-byte stores (N tiles narrower than 64 channels per pixel) ----
#pragma unroll 1
        for (int c = 0; c < BN; c += 32)
          chunk(c, [&](int g, const int4& o) {
            const int64_t off = (c + g * 8 < BN) ? elem_off(n0 + c + g * 8, out_channels) : (int64_t)-1;
            if (off >= 0) *reinterpret_cast<int4*>(outp + off) = o;
          });
      }
      if (!released) release_acc();
      if (dbg) { dbg_acc[6] += clk() - _te; dbg_acc[7] += 1; }
    }
    if (p.tma_store && q == 2 && lane == 0) bulk_wait_all();  // smem must outlive the last stores
    if (out_f32 && lane == 0) bulk_wait_all();                 // (fused head: every warp issues its own bulk copies)
  }

  if (dbg && lane == 0 && (warp == 0 || warp == 1 || warp == 2 || warp == 6)) {
    unsigned long long* o = dbg + (size_t)blockIdx.x * 24;
    if (warp == 0) { o[0] = dbg_acc[0]; o[8] = clk() - dbg_start; }
    if (warp == 1) { o[1] = dbg_acc[1]; o[2] = dbg_acc[2]; o[9] = clk() - dbg_start; }
    if (warp == 2) { for (int i = 3; i < 8; ++i) o[i] = dbg_acc[i]; o[10] = clk() - dbg_start; }
    if (warp == 6) { for (int i = 3; i < 8; ++i) o[8 + i] = dbg_acc[i]; }
  }
  // teardown
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(p.tmem_cols) : "memory");
  }
#undef FULL_BAR
#undef EMPTY_BAR
#undef TFULL_BAR
#undef TEMPTY_BAR
#undef BRES_BAR
#undef RFULL_BAR
}

typedef void (*TcKernelFn)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const TcParams, const int);

// ---------------------------------------------------------------------------------------------------------------
// Instantiations.  ~160 kernels: the build compiles this file once per PART (-DPCLS_TC_PART=k, pclsegmentation_b200/
// build.py) so that they compile in parallel; part 0 also holds the host code.  Without the macro (a plain `nvcc -c`)
// everything lands in one translation unit.
//   parts 1-8   generic kernels (RM = 0) of one (type, RES, LEAKY) combination each
//   parts 9-12  RM = 2: no residual, 16-bit outputs through the TMA-store epilogue (the float32 logits / fused-head path
//               and the direct-store path compiled out), one (type, LEAKY) combination each
//   part 0      RM = 1 (one TMA-loaded skip tensor, TMA store, ReLU: the FireDeconv expands) and the K-skip kernels
// ---------------------------------------------------------------------------------------------------------------
#ifndef PCLS_TC_PART
#define PCLS_TC_PART -1
#endif
template <typename T, bool RES, bool LEAKY>
TcKernelFn tc_kernel_for_t(int KC, int SUB, int G) {
  if (G == 4) return SUB == 3 ? conv_tc_kernel<T, 64, 3, 4, RES, LEAKY> : conv_tc_kernel<T, 64, 1, 4, RES, LEAKY>;
  if (G == 2) {
    if (KC == 64) return SUB == 3 ? conv_tc_kernel<T, 64, 3, 2, RES, LEAKY> : conv_tc_kernel<T, 64, 1, 2, RES, LEAKY>;
    return SUB == 3 ? conv_tc_kernel<T, 32, 3, 2, RES, LEAKY> : conv_tc_kernel<T, 32, 1, 2, RES, LEAKY>;
  }
  if (SUB == 3) return KC == 64 ? conv_tc_kernel<T, 64, 3, 1, RES, LEAKY> : KC == 32 ? conv_tc_kernel<T, 32, 3, 1, RES, LEAKY> : conv_tc_kernel<T, 16, 3, 1, RES, LEAKY>;
  return KC == 64 ? conv_tc_kernel<T, 64, 1, 1, RES, LEAKY> : KC == 32 ? conv_tc_kernel<T, 32, 1, 1, RES, LEAKY> : conv_tc_kernel<T, 16, 1, 1, RES, LEAKY>;
}
// ks = UMMA K steps per chunk; the one shape with a zero-padded K tail (48 channels in a 64-channel chunk: 3x3 halo
// kernel, ReLU, no residual) has its own instantiation, every other combination issues all KC / 16 steps (a run-time
// bound or predicate in the issue loop cost the issue-bound N-split layers 30 %).
template <typename T, bool LEAKY>
TcKernelFn tc_ptma_kernel_for(int KC, int SUB, int G, int ks) {
  if constexpr (!LEAKY) {
    if (ks == 3 && KC == 64 && SUB == 3 && G == 1) return conv_tc_kernel<T, 64, 3, 1, false, false, 3, 2>;
  }
  if (G == 4) return SUB == 3 ? conv_tc_kernel<T, 64, 3, 4, false, LEAKY, 4, 2> : conv_tc_kernel<T, 64, 1, 4, false, LEAKY, 4, 2>;
  if (G == 2) {
    if (KC == 64) return SUB == 3 ? conv_tc_kernel<T, 64, 3, 2, false, LEAKY, 4, 2> : conv_tc_kernel<T, 64, 1, 2, false, LEAKY, 4, 2>;
    return SUB == 3 ? conv_tc_kernel<T, 32, 3, 2, false, LEAKY, 2, 2> : conv_tc_kernel<T, 32, 1, 2, false, LEAKY, 2, 2>;
  }
  if (SUB == 3) return KC == 64 ? conv_tc_kernel<T, 64, 3, 1, false, LEAKY, 4, 2> : KC == 32 ? conv_tc_kernel<T, 32, 3, 1, false, LEAKY, 2, 2> : conv_tc_kernel<T, 16, 3, 1, false, LEAKY, 1, 2>;
  return KC == 64 ? conv_tc_kernel<T, 64, 1, 1, false, LEAKY, 4, 2> : KC == 32 ? conv_tc_kernel<T, 32, 1, 1, false, LEAKY, 2, 2> : conv_tc_kernel<T, 16, 1, 1, false, LEAKY, 1, 2>;
}
#if PCLS_TC_PART >= 0
#if PCLS_TC_PART == 1
template TcKernelFn tc_kernel_for_t<__half, false, false>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__half, false, false>(int, int, int);
#endif
#if PCLS_TC_PART == 2
template TcKernelFn tc_kernel_for_t<__half, false, true>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__half, false, true>(int, int, int);
#endif
#if PCLS_TC_PART == 3
template TcKernelFn tc_kernel_for_t<__half, true, false>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__half, true, false>(int, int, int);
#endif
#if PCLS_TC_PART == 4
template TcKernelFn tc_kernel_for_t<__half, true, true>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__half, true, true>(int, int, int);
#endif
#if PCLS_TC_PART == 5
template TcKernelFn tc_kernel_for_t<__nv_bfloat16, false, false>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__nv_bfloat16, false, false>(int, int, int);
#endif
#if PCLS_TC_PART == 6
template TcKernelFn tc_kernel_for_t<__nv_bfloat16, false, true>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__nv_bfloat16, false, true>(int, int, int);
#endif
#if PCLS_TC_PART == 7
template TcKernelFn tc_kernel_for_t<__nv_bfloat16, true, false>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__nv_bfloat16, true, false>(int, int, int);
#endif
#if PCLS_TC_PART == 8
template TcKernelFn tc_kernel_for_t<__nv_bfloat16, true, true>(int, int, int);
#else
extern template TcKernelFn tc_kernel_for_t<__nv_bfloat16, true, true>(int, int, int);
#endif
#if PCLS_TC_PART == 9
template TcKernelFn tc_ptma_kernel_for<__half, false>(int, int, int, int);
#else
extern template TcKernelFn tc_ptma_kernel_for<__half, false>(int, int, int, int);
#endif
#if PCLS_TC_PART == 10
template TcKernelFn tc_ptma_kernel_for<__half, true>(int, int, int, int);
#else
extern template TcKernelFn tc_ptma_kernel_for<__half, true>(int, int, int, int);
#endif
#if PCLS_TC_PART == 11
template TcKernelFn tc_ptma_kernel_for<__nv_bfloat16, false>(int, int, int, int);
#else
extern template TcKernelFn tc_ptma_kernel_for<__nv_bfloat16, false>(int, int, int, int);
#endif
#if PCLS_TC_PART == 12
template TcKernelFn tc_ptma_kernel_for<__nv_bfloat16, true>(int, int, int, int);
#else
extern template TcKernelFn tc_ptma_kernel_for<__nv_bfloat16, true>(int, int, int, int);
#endif
#endif  // PCLS_TC_PART >= 0

#if PCLS_TC_PART <= 0   // ---- host side + the special kernels: part 0 (or the single translation unit) ----
template <typename T>
static TcKernelFn tc_kernel_for_tt(int KC, int SUB, int G, int res, int leaky) {
  if (res) return leaky ? tc_kernel_for_t<T, true, true>(KC, SUB, G) : tc_kernel_for_t<T, true, false>(KC, SUB, G);
  return leaky ? tc_kernel_for_t<T, false, true>(KC, SUB, G) : tc_kernel_for_t<T, false, false>(KC, SUB, G);
}
static bool tc_kskip_kernel(int KC, int SUB, int G, int res, int leaky, int ks) {
  return ks == 3 && KC == 64 && SUB == 3 && G == 1 && !res && !leaky;
}
// the compile-time specialised residual kernel (RM = 1) exists for the shapes of SqueezeSegV2's FireDeconv expands
static bool tc_rtma_kernel(int KC, int SUB, int G, int res, int leaky, int rtma) {
  return rtma == 1 && res && KC == 64 && SUB == 3 && (G == 1 || G == 2 || G == 4);
}
template <typename T, bool LEAKY>
static TcKernelFn tc_rtma_kernel_for(int G) {
  if (G == 4) return conv_tc_kernel<T, 64, 3, 4, true, LEAKY, 4, 1>;
  if (G == 2) return conv_tc_kernel<T, 64, 3, 2, true, LEAKY, 4, 1>;
  return conv_tc_kernel<T, 64, 3, 1, true, LEAKY, 4, 1>;
}
static TcKernelFn tc_kernel_for(int KC, int SUB, int G, int is_bf16, int res, int leaky, int ks = 0, int rtma = 0) {
  if (rtma == 3)   // the skip computed from the network input (Net::tc_skip_fusable)
    return is_bf16 ? conv_tc_kernel<__nv_bfloat16, 64, 3, 4, true, false, 4, 3> : conv_tc_kernel<__half, 64, 3, 4, true, false, 4, 3>;
  if (rtma == 2 && !res) {
    if (is_bf16) return leaky ? tc_ptma_kernel_for<__nv_bfloat16, true>(KC, SUB, G, ks) : tc_ptma_kernel_for<__nv_bfloat16, false>(KC, SUB, G, ks);
    return leaky ? tc_ptma_kernel_for<__half, true>(KC, SUB, G, ks) : tc_ptma_kernel_for<__half, false>(KC, SUB, G, ks);
  }
  if (tc_rtma_kernel(KC, SUB, G, res, leaky, rtma)) {
    if (is_bf16) return leaky ? tc_rtma_kernel_for<__nv_bfloat16, true>(G) : tc_rtma_kernel_for<__nv_bfloat16, false>(G);
    return leaky ? tc_rtma_kernel_for<__half, true>(G) : tc_rtma_kernel_for<__half, false>(G);
  }
  if (tc_kskip_kernel(KC, SUB, G, res, leaky, ks))
    return is_bf16 ? conv_tc_kernel<__nv_bfloat16, 64, 3, 1, false, false, 3> : conv_tc_kernel<__half, 64, 3, 1, false, false, 3>;
  return is_bf16 ? tc_kernel_for_tt<__nv_bfloat16>(KC, SUB, G, res, leaky) : tc_kernel_for_tt<__half>(KC, SUB, G, res, leaky);
}

struct TcPlan {
  CUtensorMap map_a, map_b, map_c, map_r, map_b2, map_c2;
  TcParams prm;
  size_t smem_bytes;
  void* w_dev;       // plan-owned copies with permuted rows (N-split across CTAs of a merged Fire expand), else NULL
  float* bias_dev;
  ~TcPlan() { if (w_dev) cudaFree(w_dev); if (bias_dev) cudaFree(bias_dev); }
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)sym;
  }
  return fn;
}

int make_map(CUtensorMap* map, bool bf16, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                    const uint32_t* box, int swizzle_bytes) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return PCLS_ERR_CUDA; }
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                              : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, base,
                  gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r, rank); return PCLS_ERR_CUDA; }
  return PCLS_OK;
}

const int tc_debug_compiled = PCLS_TC_DEBUG;
unsigned long long* tc_debug_buf = nullptr;  // [148][24] counters of the most recent launch when enabled

// Which layers run on tensor cores: the input tensor must carry >= 16 real channels (the 6-channel network input
// goes through the CUDA-core kernel), and a stride-2 conv needs an even input width (pair view).
static bool tc_eligible(const ConvParams& p) {
  if (p.in_channels < 16 || p.cin_pad > p.in_channels) return false;
  if (p.mode == MODE_3x3_S2 && (p.Win % 2 != 0 || p.pad_left != 0)) return false;
  if (p.cout_pad > 256 && p.cout_pad % 256 != 0) return false;
  return true;
}

// Pixel-group view for narrow inputs (Cin = 16 / 32): TMA moves about one box row per ~8 cycles whatever its
// width, so G adjacent pixels are viewed as ONE row of G*Cin channels (<= 128 bytes) and the MMAs are issued
// banded (kernel comment).  Needs the whole tensor row to be contiguous (Cin == tensor channels).
static int tc_group_size(const ConvParams& cp) {
  if ((cp.mode == MODE_1x1 || cp.mode == MODE_3x3_S1 || cp.mode == MODE_ROW3) &&
      (cp.cin_pad == 16 || cp.cin_pad == 32) && cp.in_channels == cp.cin_pad && cp.cout == cp.cout_pad && !cp.out_f32 &&
      cp.Wout == cp.Win) {
    for (int g = 64 / cp.cin_pad; g >= 2; g /= 2)
      if (cp.Win % g == 0 && cp.Win / g >= 128 && g * cp.cout_pad <= 256 && (cp.cout_pad & (cp.cout_pad - 1)) == 0) return g;
  }
  return 1;
}

// Skip fusion (Net::finalize): P = 1x1 conv of the network input (<= 6 channels, no activation, no residual) whose output
// E adds as its only residual.  E computes P in its epilogue (RM = 3 kernel) when E is planned on the RM = 1 path with the
// G = 4 pixel-group view: 3x3 stride 1, 16 -> 64 channels, ReLU, TMA-store epilogue with 64-channel blocks.  Decided here,
// before the arena is planned (P's output is then never allocated); tc_plan_layer checks that the plan agrees.
bool Net::tc_skip_fusable(const ConvLayer& P, const ConvLayer& E) const {
  const ConvParams &pp = P.p, &e = E.p;
  if (P.in != 0 || pp.mode != MODE_1x1 || pp.act != PCLS_ACT_NONE || P.res0 >= 0 || P.res1 >= 0 ||
      pp.out_f32 || pp.out_coff != 0 || P.cin_logical > 6 || pp.cout != 64 || pp.out_channels != 64)
    return false;
  if (E.res0 != P.out || E.res1 >= 0 || E.in == P.out || E.pair_view || e.mode != MODE_3x3_S1 || e.act != PCLS_ACT_RELU ||
      e.out_f32 || e.cout != 64 || e.res0_channels != 64)
    return false;
  if (!tc_eligible(e) || tc_group_size(e) != 4 || (e.out_channels * 2) % 16 != 0)
    return false;
  return true;
}

int Net::tc_plan_layer(ConvLayer& L, bool allow_group, bool* retry) {
  const int max_smem = 227 * 1024;
    ConvParams& cp = L.pair_view ? L.ptc : L.p;
    L.tc_ok = false;
    *retry = false;
    if (!tc_eligible(cp)) return PCLS_OK;
    TcPlan* plan = new TcPlan();
    memset(plan, 0, sizeof(TcPlan));
    TcParams& q = plan->prm;
    const bool bf16 = precision == PCLS_BF16;
    // K chunk / swizzle: the widest of 64/32/16 channels that divides cin_pad
    q.KC = (cp.cin_pad % 64 == 0) ? 64 : (cp.cin_pad % 32 == 0) ? 32 : 16;
    q.kchunks = cp.cin_pad / q.KC;
    q.ksteps = q.KC / 16;
    q.BN = cp.cout_pad <= 256 ? cp.cout_pad : 256;
    q.n_nt = cp.cout_pad / q.BN;
    const int G = allow_group ? tc_group_size(cp) : 1;
    const bool skip = L.skip_src >= 0;   // residual0 computed from the network input (RM = 3 kernel)
    const int cin_blk = cp.cin_pad;
    q.G = G; q.cout_blk = G > 1 ? cp.cout_pad : (1 << 30);
    q.cout_blk_shift = 0;
    while ((1 << q.cout_blk_shift) < q.cout_blk && q.cout_blk_shift < 30) ++q.cout_blk_shift;
    if (G > 1) { q.KC = G * cin_blk; q.kchunks = 1; q.BN = G * cp.cout_pad; q.n_nt = 1; }
    const int swz = q.KC * 2;
    const int swz_b = G > 1 ? cin_blk * 2 : swz;
    // split-N: leading output channels whose kernel is zero outside the centre tap (the expand1x1 half of a merged Fire
    // expand layer).  Multiples of 16 channels on both sides (UMMA N granularity at M = 128).
    q.n1 = 0;
    if (G == 1 && cp.mode == MODE_3x3_S1 && q.n_nt == 1 && !L.pair_view) {
      int z = 0;
      for (; z < cp.cout_pad; ++z) {
        bool zero = true;
        for (int t = 0; t < 9 && zero; ++t) {
          if (t == 4) continue;
          const float* wr = &L.w_f32[((size_t)t * cp.cout_pad + z) * cp.cin_pad];
          for (int ci = 0; ci < cp.cin_pad; ++ci) if (wr[ci] != 0.0f) { zero = false; break; }
        }
        if (!zero) break;
      }
      z = z / 16 * 16;
      if (z >= 16 && q.BN - z >= 16) q.n1 = z;
    }
    // zero-padded K tail (48 logical channels in a 64-channel chunk): the MMAs of the all-zero K steps are not issued
    if (G == 1 && q.kchunks == 1 && q.n1 == 0) q.ksteps = std::min(q.KC / 16, (cp.cin + 15) / 16);
    // N-split across CTAs: a 3x3 layer whose weights do not fit in smem next to the pipeline (fire10's merged expand: 160 KB;
    // fire6 / fire7's 64(48) -> 192 expand3x3: 216 KB) streams them from L2 for every tile - 10 x the bytes of the A tile,
    // L2 -> smem bound (wait-cycle counters: issuer 50 % on FULL).  Cutting N in two and giving every CTA one half keeps the
    // half resident; the A tiles are then loaded twice, from L2.  Merged expands ([expand1x1 | expand3x3], n1 centre-only
    // channels) are cut so that each half holds half of BOTH parts (rows permuted): equal work per CTA, split-N per half.
    q.nsplit = 0; q.perm = 0;
    for (int i = 0; i < 8; ++i) q.cblk_off[i] = i * 64;
    std::vector<int> row_perm;   // new weight row -> old weight row, when permuted
    if (G == 1 && cp.mode == MODE_3x3_S1 && q.n_nt == 1 && !L.pair_view &&
        q.KC == 64 && !cp.out_f32 && cp.cout == cp.cout_pad && cp.Wout >= 128 && L.res1 < 0) {
      const int btile1 = q.BN * q.KC * 2, bsmall1 = (q.BN - q.n1) * q.KC * 2;
      const int all_w1 = q.n1 > 0 ? q.kchunks * (btile1 + 8 * bsmall1) : 9 * q.kchunks * btile1;
      const int half = q.BN / 2;
      if (all_w1 > 112 * 1024) {
        if (q.n1 > 0 && q.n1 % 128 == 0 && (q.BN - q.n1) % 128 == 0) {
          const int h1 = q.n1 / 2, h3 = (q.BN - q.n1) / 2;
          if (q.kchunks * ((h1 + h3) * q.KC * 2 + 8 * h3 * q.KC * 2) <= 112 * 1024) {
            row_perm.resize(q.BN);
            int blk = 0;
            for (int nt = 0; nt < 2; ++nt) {
              for (int j = 0; j < h1; ++j) row_perm[nt * (h1 + h3) + j] = nt * h1 + j;
              for (int j = 0; j < h3; ++j) row_perm[nt * (h1 + h3) + h1 + j] = q.n1 + nt * h3 + j;
              for (int j = 0; j < h1; j += 64) q.cblk_off[blk++] = nt * h1 + j;
              for (int j = 0; j < h3; j += 64) q.cblk_off[blk++] = q.n1 + nt * h3 + j;
            }
            q.BN = h1 + h3; q.n_nt = 2; q.n1 = h1; q.nsplit = 1; q.perm = 1;
          }
        } else if (q.n1 == 0 && half % 32 == 0 && 9 * q.kchunks * half * q.KC * 2 <= 112 * 1024) {
          q.BN = half; q.n_nt = 2; q.nsplit = 1;
        }
      }
    }
    q.b_small_bytes = (q.BN - q.n1) * q.KC * 2;
    // pixel grid tiled by BW x BH = 128
    const bool deconv = cp.mode == MODE_DECONV;  // (two-phase form; MODE_ROW3 is the single-pass form)
    q.Hgrid = cp.H;
    q.Wgrid = deconv ? cp.Win : cp.Wout / G;
    q.Wout = cp.Wout;
    q.out_wmul = deconv ? 2 : G;
    q.n_phase = deconv ? 2 : 1;
    int bw = 128;
    while (bw > 1 && bw / 2 >= q.Wgrid) bw /= 2;  // smallest power of two >= Wgrid, capped at 128
    q.BW = bw; q.BH = 128 / bw;
    q.bw_shift = 0;
    while ((1 << q.bw_shift) < bw) ++q.bw_shift;
    q.n_wt = (q.Wgrid + q.BW - 1) / q.BW;
    q.n_ht = (q.Hgrid + q.BH - 1) / q.BH;
    q.num_tiles = q.n_nt * q.n_phase * q.n_wt * q.n_ht;  // per frame
    // K walk
    q.a_is_5d = cp.mode == MODE_3x3_S2 ? 1 : 0;
    q.sub = 1; q.a_rows = 128;
    // halo reuse needs the three weight tiles of a row next to the A tile: only when >= 4 stages still fit
    bool halo = (cp.mode == MODE_3x3_S1 || cp.mode == MODE_ROW3) && q.BW == 128;
    if (halo) {
      const int btile_ = G > 1 ? cp.cout_pad * cin_blk * 2 : q.BN * q.KC * 2;
      const int all_w_ = q.n1 > 0 ? q.kchunks * (btile_ + (cp.ntaps - 1) * q.b_small_bytes) : cp.ntaps * q.kchunks * btile_;
      const bool resident_ = (q.n_nt == 1 || q.nsplit) && all_w_ <= 112 * 1024;
      const int st_ = (130 * q.KC * 2 + 1023) / 1024 * 1024 + (resident_ ? 0 : 3 * btile_);
      // (N-split layers hold half of a big weight set: they take two staging buffers per group instead of three)
      const int staging_ = 2 * TC_NG * 16384 + ((L.res0 >= 0 && (q.BN <= 128 || resident_) && !q.nsplit) ? TC_NG * 16384 : 0);
      if ((max_smem - 2048 - staging_ - cp.cout_pad * 4 - (resident_ ? all_w_ + 1024 : 0)) / st_ < 3) halo = false;
    }
    if (G > 1 && cp.mode != MODE_1x1 && !halo) {  // the banded issue of a 3-tap row needs the halo tile: plan again ungrouped
      delete plan;
      *retry = true;
      return PCLS_OK;
    }
    if (cp.mode == MODE_1x1) {
      q.n_groups = 1;
    } else if (halo && cp.mode == MODE_3x3_S1) {
      // one A tile of 130 pixels (one-pixel halo each side, zero-filled by TMA at the image border) per input row
      // serves the three horizontal taps: tap dw starts (dw + 1) rows into the tile.
      q.n_groups = 3; q.sub = 3; q.a_rows = 130;
      for (int g = 0; g < 3; ++g) {
        q.grp_dh[0][g] = g - 1; q.grp_dw[0][g] = -1;
        for (int u = 0; u < 3; ++u) q.grp_w[0][g][u] = g * 3 + u;
      }
      q.sub_row[0] = 0; q.sub_row[1] = 1; q.sub_row[2] = 2;
    } else if (halo && cp.mode == MODE_ROW3) {
      q.n_groups = 1; q.sub = 3; q.a_rows = 130;
      q.grp_dh[0][0] = 0; q.grp_dw[0][0] = -1;
      for (int u = 0; u < 3; ++u) { q.grp_w[0][0][u] = u; q.sub_row[u] = u; }
    } else if (cp.mode == MODE_ROW3) {
      q.n_groups = 3;
      for (int t = 0; t < 3; ++t) { q.grp_dh[0][t] = 0; q.grp_dw[0][t] = t - 1; q.grp_w[0][t][0] = t; }
    } else if (cp.mode == MODE_3x3_S1) {
      q.n_groups = 9;
      for (int t = 0; t < 9; ++t) { q.grp_dh[0][t] = t / 3 - 1; q.grp_dw[0][t] = t % 3 - 1; q.grp_w[0][t][0] = t; }
    } else if (cp.mode == MODE_PAIR6) {
      q.n_groups = 6;  // pixel-pair view of the 8-channel input: pair wo holds kx = 0,1; pair wo + 1 holds kx = 2
      for (int t = 0; t < 6; ++t) { q.grp_dh[0][t] = t / 2 - 1; q.grp_dw[0][t] = t % 2; q.grp_w[0][t][0] = t; }
    } else if (cp.mode == MODE_3x3_S2) {
      q.n_groups = 9;  // input column 2*wo + kx -> (parity kx & 1, pair wo + (kx >> 1))
      for (int t = 0; t < 9; ++t) {
        q.grp_dh[0][t] = t / 3 - 1; q.grp_par[0][t] = (t % 3) & 1; q.grp_dw[0][t] = (t % 3) >> 1; q.grp_w[0][t][0] = t;
      }
    } else {
      q.n_groups = 2;  // out[2j]   = in[j] w1 + in[j-1] w3 ;  out[2j+1] = in[j+1] w0 + in[j] w2
      q.grp_dw[0][0] = 0;  q.grp_w[0][0][0] = 1;
      q.grp_dw[0][1] = -1; q.grp_w[0][1][0] = 3;
      q.grp_dw[1][0] = 1;  q.grp_w[1][0][0] = 0;
      q.grp_dw[1][1] = 0;  q.grp_w[1][1][0] = 2;
    }
    // TMA-store epilogue: 16-bit outputs whose N tile splits into blocks of <= 64 channels
    q.tma_store = 0; q.cbw = 0; q.c_stage_bytes = 0; q.c_is_5d = (deconv || G > 1) ? 1 : 0;
    // (measured: for N tiles narrower than 64 channels the direct 16-byte stores are faster than staging)
    // (N tile = 64 k + 32, e.g. the halves of fire6 / fire7's 192-channel expand3x3: the tail block is stored through a
    // second map with 64-byte rows - with per-thread stores that epilogue took 50 cycles per column instead of 24)
    const bool narrow_tail = q.BN % 64 == 32 && q.BN > 64 && G == 1 && !deconv && L.res0 < 0 && L.res1 < 0;
    if (!cp.out_f32 && cp.cout == cp.cout_pad && (q.BN % 64 == 0 || narrow_tail) &&
        (G == 1 || cp.cout_pad % 64 == 0) &&
        (cp.out_channels * 2) % 16 == 0) {
      q.tma_store = 1;
      q.cbw = q.BN < 64 ? q.BN : 64;
      q.c_stage_bytes = (128 * q.cbw * 2 + 1023) / 1024 * 1024;
    }
    // residual0 is staged through smem only for the memory-bound layers (N tile <= 128): the wide Darknet layers are
    // tensor-bound and keep their smem for pipeline stages
    // pipeline depth; weights stay resident in smem when the whole layer fits next to >= 4 stages
    q.a_bytes = (q.a_rows * q.KC * 2 + 1023) / 1024 * 1024;
    q.b_tile_bytes = G > 1 ? cp.cout_pad * cin_blk * 2 : q.BN * q.KC * 2;
    const int all_w = q.n1 > 0 ? q.kchunks * (q.b_tile_bytes + 8 * q.b_small_bytes)
                               : q.n_phase * q.n_groups * q.kchunks * q.sub * q.b_tile_bytes;
    q.bres_tx = all_w;
    q.b_resident = ((q.n_nt == 1 || q.nsplit) && all_w <= 112 * 1024) ? 1 : 0;
    if (q.nsplit && !q.b_resident) { set_error("tc plan: N-split layer lost its resident weights"); delete plan; return PCLS_ERR_STATE; }
    q.bres_bytes = q.b_resident ? (all_w + 1023) / 1024 * 1024 : 0;
    // residual0 of the memory-bound layers (resident weights) with the TMA-store epilogue: TMA-loaded into a third
    // staging buffer and added in place (no per-thread address arithmetic, a whole block of latency hiding)
    q.res_tma = (!skip && L.res0 >= 0 && q.tma_store && q.cbw == 64 && q.b_resident && (cp.res0_channels * 2) % 16 == 0) ? 1 : 0;
    q.n_cbuf = (q.res_tma && !q.nsplit) ? 3 : 2;
    q.res_smem = (!skip && !q.res_tma && L.res0 >= 0 && q.BN <= 128) ? 1 : 0;
    // (skip: two 8 KB network-input tiles per group in place of the third staging buffer)
    const int cstage_total = (q.tma_store ? q.n_cbuf * TC_NG * q.c_stage_bytes : 0) + ((q.res_smem || skip) ? TC_NG * 16384 : 0);
    if (skip && !(G == 4 && q.tma_store && q.cbw == 64 && q.b_resident && q.BN == 256 && q.BW == 128 && q.BH == 1)) {
      set_error("tc plan: the layer that computes the fused skip is not planned on the G = 4 TMA-store path");
      delete plan; return PCLS_ERR_STATE;
    }
    if (G > 1 && !q.b_resident) { delete plan; *retry = true; return PCLS_OK; }
    const int stage_bytes = q.a_bytes + (q.b_resident ? 0 : q.sub * q.b_tile_bytes);
    int stages = (max_smem - 2048 - cp.cout_pad * 4 - q.bres_bytes - cstage_total - (cp.out_f32 ? 4 * TC_NG * 32 * 33 * 4 : 0)) / stage_bytes;
    if (stages > 12) stages = 12;
    if (stages < 2) { delete plan; *retry = G > 1; return PCLS_OK; }
    q.stages = stages;
    plan->smem_bytes = (size_t)stages * stage_bytes + q.bres_bytes + cstage_total + 1024 /*alignment slack*/ +
                       (size_t)(2 * stages + 17 + 3 * TC_NG) * 8 + 48 + (cp.out_f32 ? 4 * TC_NG * 32 * 33 * 4 : 0) + (size_t)cp.cout_pad * 4 /*bias*/;
    // descriptors
    const uint32_t layout = swz == 128 ? 2u : swz == 64 ? 4u : 6u;  // UMMA LayoutType
    const uint32_t sbo = (uint32_t)(8 * swz) >> 4;                   // 8 rows of one swizzle span
    q.desc_hi = sbo | (1u << 14) /*descriptor version (sm_100)*/ | (layout << 29);
    {
      const uint32_t layout_b = swz_b == 128 ? 2u : swz_b == 64 ? 4u : 6u;
      q.desc_hi_b = ((uint32_t)(8 * swz_b) >> 4) | (1u << 14) | (layout_b << 29);
      q.idesc_blk = (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) |
                    ((uint32_t)(cp.cout_pad >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    }
    q.idesc = (1u << 4) /*D = f32*/ | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) |
              ((uint32_t)(q.BN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    q.idesc_small = (q.idesc & ~(0x3Fu << 17)) | ((uint32_t)((q.BN - q.n1) >> 3) << 17);
    q.idesc_lo = (q.idesc & ~(0x3Fu << 17)) | ((uint32_t)(q.n1 >> 3) << 17);
    q.n_acc = 2;
    while (q.n_acc < 8 && q.n_acc * 2 * q.BN <= 512) q.n_acc *= 2;
    uint32_t cols = 32;
    while (cols < (uint32_t)(q.n_acc * q.BN)) cols <<= 1;
    q.tmem_cols = cols;
    // epilogue
    q.cout = cp.cout; q.out_channels = cp.out_channels; q.out_coff = cp.out_coff; q.act = cp.act;
    q.out_f32 = cp.out_f32; q.is_bf16 = bf16 ? 1 : 0;
    q.res0_channels = cp.res0_channels; q.res1_channels = cp.res1_channels;
    q.bias = cp.bias;

    // tensor maps.  A: activations of the input tensor inside the arena (extent = frames_per_pass frames).
    char* a_base = (char*)tensor_ptr(L.in, frames_per_pass);
    const uint64_t C = (uint64_t)cp.in_channels * G, Wi = (uint64_t)cp.Win / G, Hh = (uint64_t)cp.H, F = (uint64_t)frames_per_pass;
    int rc;
    if (q.a_is_5d) {
      const uint64_t dims[5] = {C, 2, Wi / 2, Hh, F};
      const uint64_t str[4] = {C * 2, C * 4, Wi * C * 2, Hh * Wi * C * 2};
      const uint32_t box[5] = {(uint32_t)q.KC, 1, (uint32_t)q.BW, (uint32_t)q.BH, 1};
      rc = make_map(&plan->map_a, bf16, a_base, 5, dims, str, box, swz);
    } else {
      const uint64_t dims[4] = {C, Wi, Hh, F};
      const uint64_t str[3] = {C * 2, Wi * C * 2, Hh * Wi * C * 2};
      const uint32_t box[4] = {(uint32_t)q.KC, (uint32_t)(q.BH == 1 ? q.a_rows : q.BW), (uint32_t)q.BH, 1};
      rc = make_map(&plan->map_a, bf16, a_base, 4, dims, str, box, swz);
    }
    if (rc) { delete plan; return rc; }
    const void* w_src = cp.w;
    if (q.perm) {   // permuted copies of the packed weights [tap][row][cin_pad] and of the bias
      std::vector<uint16_t> hw((size_t)cp.ntaps * cp.cout_pad * cp.cin_pad);
      std::vector<float> hb(cp.cout_pad);
      for (int t = 0; t < cp.ntaps; ++t)
        for (int n = 0; n < cp.cout_pad; ++n)
          for (int ci = 0; ci < cp.cin_pad; ++ci) {
            const float w = L.w_f32[((size_t)t * cp.cout_pad + row_perm[n]) * cp.cin_pad + ci];
            uint16_t bits;
            if (bf16) { __nv_bfloat16 hv = __float2bfloat16_rn(w); memcpy(&bits, &hv, 2); }
            else { __half hv = __float2half_rn(w); memcpy(&bits, &hv, 2); }
            hw[((size_t)t * cp.cout_pad + n) * cp.cin_pad + ci] = bits;
          }
      for (int n = 0; n < cp.cout_pad; ++n) hb[n] = L.bias_f32[row_perm[n]];
      if (cudaMalloc(&plan->w_dev, hw.size() * 2) != cudaSuccess || cudaMalloc((void**)&plan->bias_dev, hb.size() * 4) != cudaSuccess ||
          cudaMemcpy(plan->w_dev, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess ||
          cudaMemcpy(plan->bias_dev, hb.data(), hb.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("tc plan: upload of the permuted weights failed"); delete plan; return PCLS_ERR_CUDA;
      }
      w_src = plan->w_dev;
      q.bias = plan->bias_dev;
    }
    {
      const uint64_t dims[3] = {(uint64_t)cp.cin_pad, (uint64_t)cp.cout_pad, (uint64_t)cp.ntaps};
      const uint64_t str[2] = {(uint64_t)cp.cin_pad * 2, (uint64_t)cp.cin_pad * cp.cout_pad * 2};
      const uint32_t box[3] = {(uint32_t)(G > 1 ? cin_blk : q.KC), (uint32_t)(G > 1 ? cp.cout_pad : q.BN), 1};
      rc = make_map(&plan->map_b, bf16, const_cast<void*>(w_src), 3, dims, str, box, swz_b);
    }
    if (rc) { delete plan; return rc; }
    plan->map_b2 = plan->map_b;
    if (q.n1 > 0) {  // weight rows [n1, BN) of one tap
      const uint64_t dims[3] = {(uint64_t)cp.cin_pad, (uint64_t)cp.cout_pad, (uint64_t)cp.ntaps};
      const uint64_t str[2] = {(uint64_t)cp.cin_pad * 2, (uint64_t)cp.cin_pad * cp.cout_pad * 2};
      const uint32_t box[3] = {(uint32_t)q.KC, (uint32_t)(q.BN - q.n1), 1};
      rc = make_map(&plan->map_b2, bf16, const_cast<void*>(w_src), 3, dims, str, box, swz_b);
      if (rc) { delete plan; return rc; }
    }
    if (q.tma_store) {  // C: the output tensor (or its re-viewed form) inside the arena
      char* c_base = (char*)tensor_ptr(L.out, frames_per_pass);
      const uint64_t Co = (uint64_t)cp.out_channels, Wo = (uint64_t)cp.Wout;
      const int csw = q.cbw == 64 ? 128 : 0;
      if (q.c_is_5d) {  // two-phase transposed conv: dim 1 = output column parity; pixel groups: dim 1 = pixel in group
        const uint64_t gg = G > 1 ? (uint64_t)G : 2;
        const uint64_t dims[5] = {Co, gg, Wo / gg, Hh, F};
        const uint64_t str[4] = {Co * 2, Co * 2 * gg, Wo * Co * 2, Hh * Wo * Co * 2};
        const uint32_t box[5] = {(uint32_t)q.cbw, 1, (uint32_t)q.BW, (uint32_t)q.BH, 1};
        rc = make_map(&plan->map_c, bf16, c_base, 5, dims, str, box, csw);
      } else {
        const uint64_t dims[4] = {Co, Wo, Hh, F};
        const uint64_t str[3] = {Co * 2, Wo * Co * 2, Hh * Wo * Co * 2};
        const uint32_t box[4] = {(uint32_t)q.cbw, (uint32_t)q.BW, (uint32_t)q.BH, 1};
        rc = make_map(&plan->map_c, bf16, c_base, 4, dims, str, box, csw);
      }
      if (rc) { delete plan; return rc; }
      plan->map_c2 = plan->map_c;
      if (q.BN % 64 == 32) {      // 32-channel tail block of the N tile
        const uint64_t dims[4] = {Co, Wo, Hh, F};
        const uint64_t str[3] = {Co * 2, Wo * Co * 2, Hh * Wo * Co * 2};
        const uint32_t box[4] = {32u, (uint32_t)q.BW, (uint32_t)q.BH, 1};
        rc = make_map(&plan->map_c2, bf16, c_base, 4, dims, str, box, 64);
        if (rc) { delete plan; return rc; }
      }
    } else {
      plan->map_c = plan->map_a;  // unused
      plan->map_c2 = plan->map_a;
    }
    plan->map_r = plan->map_c;
    if (skip) {
      // R: the network input viewed as rows of four pixels x 8 channels (64 bytes); a tile is 128 such rows.
      // Skip weights [64][8]: channels 0-5 of the source conv, its bias split into hi + lo (= bias - hi) in 6 and 7.
      const ConvLayer& P = convs[L.skip_src];
      const uint64_t dims[4] = {32, (uint64_t)W / 4, Hh, F};
      const uint64_t str[3] = {64, (uint64_t)W / 4 * 64, Hh * (uint64_t)W / 4 * 64};
      const uint32_t box[4] = {32, (uint32_t)q.BW, 1, 1};
      rc = make_map(&plan->map_r, bf16, tensor_ptr(P.in, frames_per_pass), 4, dims, str, box, 64);
      if (rc) { delete plan; return rc; }
      std::vector<float> ws(64 * 8, 0.0f);
      for (int n = 0; n < 64; ++n) {
        for (int ci = 0; ci < P.cin_logical; ++ci) ws[n * 8 + ci] = P.w_f32[(size_t)n * P.p.cin_pad + ci];
        const float b = P.bias_f32[n];
        const float hi = bf16 ? __bfloat162float(__float2bfloat16_rn(b)) : __half2float(__float2half_rn(b));
        ws[n * 8 + 6] = hi; ws[n * 8 + 7] = b - hi;
      }
      std::vector<uint16_t> hw(ws.size());
      for (size_t i = 0; i < ws.size(); ++i) {
        if (bf16) { __nv_bfloat16 hv = __float2bfloat16_rn(ws[i]); memcpy(&hw[i], &hv, 2); }
        else { __half hv = __float2half_rn(ws[i]); memcpy(&hw[i], &hv, 2); }
      }
      if (cudaMalloc(&plan->w_dev, hw.size() * 2) != cudaSuccess ||
          cudaMemcpy(plan->w_dev, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("tc plan: upload of the skip weights failed"); delete plan; return PCLS_ERR_CUDA;
      }
      q.skip = 1; q.skip_w = plan->w_dev;
    }
    if (q.res_tma) {  // R: the residual tensor, same view as C
      char* r_base = (char*)tensor_ptr(L.res0, frames_per_pass);
      const uint64_t Co = (uint64_t)cp.res0_channels, Wo = (uint64_t)cp.Wout;
      if (q.c_is_5d) {
        const uint64_t gg = G > 1 ? (uint64_t)G : 2;
        const uint64_t dims[5] = {Co, gg, Wo / gg, Hh, F};
        const uint64_t str[4] = {Co * 2, Co * 2 * gg, Wo * Co * 2, Hh * Wo * Co * 2};
        const uint32_t box[5] = {(uint32_t)q.cbw, 1, (uint32_t)q.BW, (uint32_t)q.BH, 1};
        rc = make_map(&plan->map_r, bf16, r_base, 5, dims, str, box, 128);
      } else {
        const uint64_t dims[4] = {Co, Wo, Hh, F};
        const uint64_t str[3] = {Co * 2, Wo * Co * 2, Hh * Wo * Co * 2};
        const uint32_t box[4] = {(uint32_t)q.cbw, (uint32_t)q.BW, (uint32_t)q.BH, 1};
        rc = make_map(&plan->map_r, bf16, r_base, 4, dims, str, box, 128);
      }
      if (rc) { delete plan; return rc; }
    }
    L.tc = plan;
    L.tc_ok = true;
  return PCLS_OK;
}

int Net::tc_prepare() {
  const int max_smem = 227 * 1024;
  static bool attr_set_dev[64] = {false};   // the opt-in to > 48 KB dynamic smem is per device (and context)
  int dev = 0;
  PCLS_CHECK_CUDA(cudaGetDevice(&dev));
  bool& attr_set = attr_set_dev[dev & 63];
  for (auto& L : convs) {
    bool retry = false;
    if (L.skip_into >= 0) continue;   // computed by the layer that reads it (no launch of its own)
    int rc = head_plan_layer(L);   // the logits layer has its own kernel (conv_head.cu); falls through when it does not qualify
    if (rc) return rc;
    if (L.hp) { L.tc_ok = true; continue; }
    rc = tc_plan_layer(L, true, &retry);
    if (rc == PCLS_OK && retry) rc = tc_plan_layer(L, false, &retry);  // pixel-group view did not fit: plan ungrouped
    if (rc) return rc;
  }
  if (!attr_set) {
    for (int kc = 16; kc <= 64; kc *= 2)
      for (int sub = 1; sub <= 3; sub += 2)
        for (int g = 1; g <= 4; g *= 2) {
          if ((g == 4 && kc != 64) || (g == 2 && kc == 16)) continue;
          for (int bf = 0; bf < 2; ++bf)
            for (int rs = 0; rs < 2; ++rs)
              for (int lk = 0; lk < 2; ++lk)
                PCLS_CHECK_CUDA(cudaFuncSetAttribute(tc_kernel_for(kc, sub, g, bf, rs, lk), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        }
    for (int bf = 0; bf < 2; ++bf) {
      PCLS_CHECK_CUDA(cudaFuncSetAttribute(tc_kernel_for(64, 3, 1, bf, 0, 0, 3), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
      for (int g = 1; g <= 4; g *= 2)
        for (int lk = 0; lk < 2; ++lk)
          PCLS_CHECK_CUDA(cudaFuncSetAttribute(tc_kernel_for(64, 3, g, bf, 1, lk, 0, 1), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
      for (int kc = 16; kc <= 64; kc *= 2)
        for (int sub = 1; sub <= 3; sub += 2)
          for (int g = 1; g <= 4; g *= 2) {
            if ((g == 2 && kc < 32) || (g == 4 && kc < 64)) continue;
            for (int lk = 0; lk < 2; ++lk)
              PCLS_CHECK_CUDA(cudaFuncSetAttribute(tc_kernel_for(kc, sub, g, bf, 0, lk, 0, 2), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
          }
      PCLS_CHECK_CUDA(cudaFuncSetAttribute(tc_kernel_for(64, 3, 1, bf, 0, 0, 3, 2), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
      PCLS_CHECK_CUDA(cudaFuncSetAttribute(tc_kernel_for(64, 3, 4, bf, 1, 0, 0, 3), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    }
    attr_set = true;
  }
  return PCLS_OK;
}

int Net::tc_launch(ConvLayer& L, const ConvParams& p, int nb, cudaStream_t s) {
  if (L.hp) return head_launch(L, p, nb, s);
  TcPlan* plan = L.tc;
  TcParams prm = plan->prm;
  prm.out = p.out; prm.res0 = p.res0; prm.res1 = p.res1;
  prm.dbg = tc_debug_buf;
  prm.pdl_early = pdl_early_now;
  prm.head = (prm.out_f32 && head_args.head) ? 1 : 0;
  prm.none_index = head_args.none_index; prm.mask = head_args.mask;
  prm.probs = head_args.probs; prm.preds = head_args.preds; prm.logits = head_args.logits;
  const int num_tiles = prm.num_tiles * nb;
  if (num_tiles == 0) return PCLS_OK;
  int grid = num_tiles < sm_count() ? num_tiles : sm_count();
  if (prm.nsplit) grid -= grid % prm.n_nt;   // every CTA sees one N tile only (tile % n_nt == blockIdx.x % n_nt)
  // one skip tensor, TMA-loaded into the staging buffers, TMA-store epilogue, ReLU: the specialised residual kernel
  const int rtma = prm.skip ? 3 : (prm.res_tma && prm.res0 && !prm.res1 && prm.tma_store && !prm.out_f32 &&
                                   (prm.act == PCLS_ACT_RELU || prm.act == PCLS_ACT_LEAKY)) ? 1
                 : (!prm.res0 && !prm.res1 && prm.tma_store && !prm.out_f32) ? 2 : 0;
  const bool res = prm.res0 || prm.res1 || prm.skip;
  PCLS_CHECK_CUDA(launch_pdl(tc_kernel_for(prm.KC, prm.sub, prm.G, prm.is_bf16, res ? 1 : 0, prm.act == PCLS_ACT_LEAKY ? 1 : 0, prm.ksteps, rtma),
                             dim3(grid), dim3(TC_THREADS), plan->smem_bytes, s,
                             plan->map_a, plan->map_b, plan->map_c, plan->map_r, plan->map_b2, plan->map_c2, prm, num_tiles));
  return check_launch("conv_tc_kernel");
}

void Net::tc_release() {
  for (auto& L : convs) { delete L.tc; L.tc = nullptr; L.tc_ok = false; head_release(L); }
}

#endif  // PCLS_TC_PART <= 0

}  // namespace pcls
