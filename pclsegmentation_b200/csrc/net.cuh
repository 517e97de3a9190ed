// Internal definition of pcls_net (the op-list executor).
#pragma once
#include <vector>

#include "nn_kernels.cuh"

namespace pcls {

struct TensorInfo {
  int width = 0, channels = 0;
  int stride = 0;             // channels per pixel in memory (>= channels: 48-channel tensors are padded to 64, see add_conv)
  bool logits = false;
  int first = -1, last = -1;  // op indices of first write / last use
  size_t offset = 0;          // per-frame byte offset inside the arena (scaled by frames_per_pass)
};

struct TcPlan;    // tcgen05 launch plan of one conv layer (conv_tc.cu)
struct HeadPlan;  // launch plan of the logits layer + fused segmentation head (conv_head.cu)
extern const int tc_debug_compiled;
extern unsigned long long* tc_debug_buf;  // wait-cycle counters of the most recent conv_tc_kernel launch ("tc_debug")

struct ConvLayer {
  ConvParams p;
  int cin_logical = 0, cout_logical = 0;   // the layer's own channel counts (p.cin_pad / p.cout may include tensor padding)
  int in = -1, out = -1, res0 = -1, res1 = -1;
  std::vector<float> w_f32;     // folded, packed [tap][cout_pad][cin_pad]
  std::vector<float> bias_f32;  // folded [cout_pad]
  bool tc_ok = false;
  TcPlan* tc = nullptr;
  HeadPlan* hp = nullptr;
  int pool_src = -1, pool_pad_left = 0;   // >= 0: this 1x1 conv reads tensor pool_src through a fused 3x3/s2 max-pool
  int up_squeeze = -1;     // transposed conv: index of the squeeze 1x1 conv computed in front of it by the same kernel (squeeze_upconv.cu)
  int fused_into_up = -1;  // that squeeze conv: index of the transposed conv that runs it (no launch of its own)
  int skip_src = -1;       // >= 0: residual0 is that conv's output, computed in this conv's epilogue from its input (conv_tc.cu, RM = 3)
  int skip_into = -1;      // that conv: index of the conv that computes it (no launch, its output tensor is never allocated)
  // Pixel-pair view for the convolutions that read the 8-channel network input (tensor-core path only):
  // [B,H,W,8] is viewed as [B,H,W/2,16]; `ptc` / `w_tc` / `bias_tc` describe the equivalent convolution on pairs.
  bool pair_view = false;
  ConvParams ptc;
  std::vector<float> w_tc, bias_tc;
  void* w_tc_dev = nullptr;
  float* bias_tc_dev = nullptr;
};

struct PoolLayer { int in, out, pad_left; int fused_conv = -1; /* index of the 1x1 conv that pools on the fly (pool_conv.cu), -1: own kernel */ };

struct CamLayer {
  int in, out, C, R;
  std::vector<float> h;  // w1 [C][R], w2 [R][C], b1 [R], b2 [C]
  CamParams p;
};

// In-place MC dropout of one tensor (mc_dropout.cu); only in a net built with pcls_net_dropout.
struct DropoutLayer { int tensor, site; uint32_t thr; float scale; };

enum OpType { OP_CONV = 0, OP_POOL = 1, OP_CAM = 2, OP_DROPOUT = 3 };
struct OpRef { int type, index; };

constexpr int kIn16 = 0x100;   // OR-ed into `channels` inside the library: the input is 16-bit (pcls_net_forward_in16)

struct GraphKey {
  const void *lidar, *mask, *logits, *probs, *preds;
  int channels, B, raw, conv_impl;
  double norm[10];
};
struct CachedGraph { GraphKey key; cudaGraphExec_t exec = nullptr; uint64_t stamp = 0; };

struct Net {
  int H = 0, W = 0, precision = PCLS_F16, max_batch = 0;
  std::vector<TensorInfo> tensors;
  std::vector<ConvLayer> convs;
  std::vector<PoolLayer> pools;
  std::vector<CamLayer> cams;
  std::vector<DropoutLayer> dropouts;
  std::vector<OpRef> ops;
  bool finalized = false;
  int logits_tensor = -1, num_classes = 0, none_index = 0;
  // execution knobs
  int conv_impl = 0;
  bool use_graph = true;
  bool fuse_up = true;     // FireDeconv squeeze 1x1 + transposed conv as one kernel (squeeze_upconv.cu)
  bool fuse_pool = true;   // max-pool + the squeeze 1x1 conv that consumes it as one kernel (pool_conv.cu)
  bool fuse_head = true;   // run softmax/argmax/mask in the epilogue of the final convolution (tcgen05 path)
  bool fuse_skip = true;   // a 1x1 conv of the network input whose only reader adds it as a skip: computed by that reader
  struct HeadArgs { int head = 0, none_index = 0; const uint8_t* mask = nullptr; float* probs = nullptr; int32_t* preds = nullptr; float* logits = nullptr; } head_args;
  int micro_batch = 0;
  bool keep_tensors = false;  // test aid: no arena reuse, every intermediate stays readable after the forward
  // device state
  int frames_per_pass = 0;
  size_t frame_bytes = 0, mask_offset = 0;
  void* arena = nullptr;
  size_t arena_bytes = 0;
  void* weights = nullptr;
  size_t weight_bytes = 0;
  int last_B = 0;
  std::vector<CachedGraph> graphs;
  uint64_t graph_clock = 0;
  int graph_misses = 0;       // consecutive forwards whose argument set was not in the graph cache
  cudaStream_t cap_stream = nullptr;
  DropState* drop_state = nullptr;   // (seed, frame_base, pass) of the dropout ops, written by pcls_net_set_dropout

  ~Net();
  int add_tensor(int width, int channels, bool logits);
  size_t tensor_frame_bytes(const TensorInfo& t) const;
  int add_conv(const pcls_conv_desc& d);
  void build_pair_view(ConvLayer& L);
  void build_deconv_row3(ConvLayer& L);
  int add_pool(int in, int out);
  int add_cam(const pcls_cam_desc& d);
  int add_dropout(int tensor, int site, double rate);
  void op_tensors(const OpRef& op, std::vector<int>& reads, std::vector<int>& writes) const;
  int finalize(int logits_tensor, int num_classes, int none_index);
  void* tensor_ptr(int t, int frames) const;
  template <typename T>
  int run_pass(const float* lidar, int channels, const uint8_t* mask, bool raw, const double* mean5, const double* std5,
               int b0, int nb, float* logits, float* probs, int32_t* preds, cudaStream_t s, cudaEvent_t* ev);
  int run_all(const float* lidar, int channels, const uint8_t* mask, bool raw, const double* mean5, const double* std5,
              int B, float* logits, float* probs, int32_t* preds, cudaStream_t s, cudaEvent_t* ev);
  void drop_graphs();
  int profile_ops(const float* lidar, int channels, const uint8_t* mask, const double* mean5, const double* std5, int B,
                  float* logits, float* probs, int32_t* preds, float* h_ms, cudaStream_t s);
  bool head_is_fused() const;
  int op_info(int i, char* name, int* family, int64_t* flops, int64_t* bytes) const;
  int forward(const float* lidar, int channels, const uint8_t* mask, const double* mean5, const double* std5, int B,
              float* logits, float* probs, int32_t* preds, cudaStream_t s);
  int read_tensor(int t, int B, float* out, cudaStream_t s);

  // tcgen05 implicit-GEMM path (conv_tc.cu)
  int tc_prepare();
  int tc_plan_layer(ConvLayer& L, bool allow_group, bool* retry);
  bool tc_skip_fusable(const ConvLayer& P, const ConvLayer& E) const;
  int tc_launch(ConvLayer& L, const ConvParams& p, int nb, cudaStream_t s);
  void tc_release();
  // logits layer + fused head (conv_head.cu)
  int head_plan_layer(ConvLayer& L);
  int head_launch(ConvLayer& L, const ConvParams& p, int nb, cudaStream_t s);
  void head_release(ConvLayer& L);
};

}  // namespace pcls
