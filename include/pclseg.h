/*
 * pclseg.h - C ABI of libpclseg.so: the B200 (sm_100a) implementation of the
 * PCLSegmentation inference hot path.
 *
 * The reference (ika-rwth-aachen/PCLSegmentation) is pure Python on numpy + TensorFlow and has
 * no FFI of its own; its "plugin boundary" for this path is the Python call contract
 *     LaserScan(project,H,W,fov_up,fov_down).set_points(...)        dataset_convert/laserscan_semantic_kitti.py:9-104
 *     SemLaserScan.set_label(...)                                    dataset_convert/laserscan_semantic_kitti.py:238-258
 *     model = SqueezeSegV2(mc) / Darknet(mc); model([lidar, mask])   pcl_segmentation/utils/args_loader.py:52-55, inference.py:75, eval.py:47
 *     tf.metrics.MeanIoU(NC).update_state(label, pred) / total_cm    pcl_segmentation/eval.py:41-58
 * Each entry point below names the reference code it replaces.  The Python mirror of that
 * contract (pclsegmentation_b200/) binds these symbols with ctypes; INTEGRATION.md shows the stub
 * a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name starts with "h_" (host);
 *   - the caller owns every input / output buffer; a pcls_net owns only its folded weights and its
 *     activation workspace (allocated in pcls_net_finalize, never inside pcls_net_forward);
 *   - all work is enqueued asynchronously on the given stream (a cudaStream_t passed as void*);
 *   - functions return 0 on success or a negative pcls_status; pcls_last_error() returns a
 *     thread-local message for the last failure on the calling thread;
 *   - a pcls_net is not thread-safe: one handle + one stream per GPU.
 *   - there is no CPU fallback anywhere: without a CUDA device every compute call fails.
 */
#ifndef PCLSEG_H_
#define PCLSEG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PCLS_ABI_VERSION 2

typedef enum pcls_status {
  PCLS_OK = 0,
  PCLS_ERR_INVALID = -1, /* bad argument / unsupported shape */
  PCLS_ERR_CUDA = -2,    /* CUDA runtime / driver error */
  PCLS_ERR_STATE = -3,   /* call order violated (e.g. forward before finalize) */
  PCLS_ERR_NCCL = -4     /* NCCL unavailable or failed */
} pcls_status;

typedef void* pcls_stream; /* cudaStream_t */

int pcls_abi_version(void);
const char* pcls_last_error(void);

/* =====================================================================================
 * Spherical projection
 * ===================================================================================== */

/* Replaces LaserScan.do_range_projection (laserscan_semantic_kitti.py:106-166, identical copy at
 * laserscan_nuscenes.py:226-286) and, when `ring` is non-NULL, do_range_projection_ring
 * (laserscan_nuscenes.py:191-223), for a BATCH of scans.
 *
 *   points   [total,4] f32  x,y,z,remission per point (the KITTI .bin record, :73-79)
 *   ring     [total] i32 or NULL.  non-NULL selects the ring variant: row = H-1-ring,
 *            winner of a pixel = highest point index (plain in-order scatter); fov is ignored.
 *   offsets  [B+1] i64: scan b owns points offsets[b] .. offsets[b+1]-1; point indices written to
 *            proj_idx are LOCAL to their scan (what the reference's per-scan loop produces).
 *   keys     [B,H,W] u64 caller-provided scratch; on return key = (bits(depth) << 32) | local index
 *            of the winning point, ~0 for an empty pixel.
 *   proj_x, proj_y [total] i32, unproj_range [total] f32: per-point outputs (:141,:146,:149); any
 *            may be NULL.  Points with a non-finite pixel coordinate (zero depth, NaN; the
 *            reference raises on those) are dropped and get proj_x = proj_y = -1.
 *
 * Arithmetic: unfused float32 exactly as numpy evaluates the reference (SURVEY.md Appendix E);
 * atan2/asin are evaluated in float64 and rounded once to float32 (correctly rounded), the tie
 * rule on equal depth is "lowest point index".  fov_*_deg are the Python doubles of the reference
 * constructor. */
int pcls_project_scatter(const float* points, const int32_t* ring, const int64_t* offsets, int B,
                         int64_t total_points, int H, int W, double fov_up_deg, double fov_down_deg,
                         uint64_t* keys, int32_t* proj_x, int32_t* proj_y, float* unproj_range,
                         pcls_stream stream);

/* Second pass: turns the winner keys into images.  Replaces the four fancy-index scatters
 * (laserscan_semantic_kitti.py:162-165), SemLaserScan.do_label_projection (:269-279; sem = label &
 * 0xFFFF) and the converter assembly (dataset_convert/semantic_kitti.py:162-173).
 *
 *   labels     [total] u32 or NULL        raw .label words
 *   label_lut  [lut_len] i32 or NULL      learning_map as a dense LUT (semantic-kitti.yaml:109-143);
 *                                         ids >= lut_len map to 0
 *   empty_fill value of x,y,z,remission,range at empty pixels: -1 = LaserScan attributes (:23-40),
 *              0 = converter output (semantic_kitti.py:162-165)
 *   image      [B,H,W,6] f32 (x,y,z,remission,range,label) or NULL.  The label channel holds
 *              LUT[sem] (LUT[0] at empty pixels) as a float, like the converter's concat.
 *   proj_idx   [B,H,W] i32 (-1 empty) or NULL
 *   proj_sem_label [B,H,W] i32 raw semantic id (0 empty) or NULL */
int pcls_project_resolve(const float* points, const uint32_t* labels, const int64_t* offsets, int B,
                         int H, int W, const uint64_t* keys, const int32_t* label_lut, int lut_len,
                         float empty_fill, float* image, int32_t* proj_idx, int32_t* proj_sem_label,
                         pcls_stream stream);

/* Fused scan -> labels pipeline (dataset_convert/semantic_kitti.py:152-173 + inference.py:47-78 without the [H,W,6] file
 * in between): turns the winner keys straight into the NETWORK INPUT - per pixel the winning point's x, y, z, remission,
 * range, masked (range > 0) and normalised in float64 with h_mean5 / h_std5 like inference.py:50-62, stored as the
 * 16-bit [B,H,W,8] pixel (5 channels + mask + 2 zeros) and the u8 mask that pcls_net_forward reads.  `input8` / `mask`
 * are the net's own buffers (pcls_net_input_buffers); then call pcls_net_forward(net, NULL, 0, NULL, NULL, NULL, B, ...).
 * precision = the net's (PCLS_F16 | PCLS_BF16); proj_idx [B,H,W] i32 or NULL. */
int pcls_project_resolve_net_input(const float* points, const int64_t* offsets, int B, int H, int W,
                                   const uint64_t* keys, const double* h_mean5, const double* h_std5, int precision,
                                   void* input8, uint8_t* mask, int32_t* proj_idx, pcls_stream stream);

/* =====================================================================================
 * Segmentation head, input stage, confusion matrix
 * ===================================================================================== */

/* Replaces PCLSegmentationNetwork.segmentation_head (nets/SegmentationNetwork.py:58-69):
 * probabilities = softmax(logits); predictions = argmax(probabilities) (lowest index on ties, taken
 * over the rounded float32 probabilities) ; predictions = none_index where mask == 0.
 *   logits [n_pixels,NC] f32, mask [n_pixels] u8 (bool) or NULL, probs [n_pixels,NC] f32 or NULL,
 *   preds [n_pixels] i32.  NC <= 32. */
int pcls_head(const float* logits, const uint8_t* mask, int64_t n_pixels, int num_classes,
              int none_index, float* probs, int32_t* preds, pcls_stream stream);

/* Replaces the input stage inference.py:47-72 == DataLoader.parse_sample (data_loader.py:153-187):
 * mask = depth > 0; (x - INPUT_MEAN) / INPUT_STD in float64; zero where ~mask; append mask; the label fix-up
 * label[~mask] = none_index; and the class-weight map weight[label == l] = CLS_LOSS_WEIGHT[l] (:181-185).
 *   sample  [n_pixels, channels] f32, channels = 5 (x,y,z,i,d) or 6 (+label)
 *   h_mean5 / h_std5  host doubles (mc.INPUT_MEAN / mc.INPUT_STD)
 *   lidar   [n_pixels,6] f32 or NULL; mask [n_pixels] u8 or NULL; label [n_pixels] i32 or NULL
 *   h_cls_loss_weight  host doubles [num_classes] (mc.CLS_LOSS_WEIGHT) or NULL; weight [n_pixels] f32 or NULL: 0 where
 *           the label is not one of 0 .. num_classes-1 (the reference starts from np.zeros), num_classes <= 32
 *           (label and weight require channels == 6). */
int pcls_input_stage(const float* sample, int channels, int64_t n_pixels, const double* h_mean5,
                     const double* h_std5, int none_index, float* lidar, uint8_t* mask,
                     int32_t* label, const double* h_cls_loss_weight, int num_classes, float* weight,
                     pcls_stream stream);

/* float64 -> float32 narrowing on the device (round to nearest even), for the float64 `[H,W,6]` range-image files
 * the reference's converters write (dataset_convert/semantic_kitti.py:173) and inference.py:47 / the data loader cast
 * on the host.  in: n doubles (16-byte aligned), out: n floats. */
int pcls_cast_f64_f32(const double* in, float* out, int64_t n, pcls_stream stream);

/* nuScenes LiDAR records on the device: `rec5` [n,5] f32 (x, y, z, intensity, ring index - the 5-float .bin record of
 * dataset_convert/laserscan_nuscenes.py:27-28, split at :139-145) -> `points4` [n,4] f32 (x,y,z,remission, 16-byte aligned),
 * the layout pcls_project_scatter reads, and `ring` [n] i32 (= astype(np.int32); may be NULL).  KITTI .bin files are
 * already [n,4] records and need no unpacking. */
int pcls_unpack_xyzir(const float* rec5, int64_t n, float* points4, int32_t* ring, pcls_stream stream);

/* Replaces tf.keras.metrics.MeanIoU.update_state (eval.py:41,48; tf.math.confusion_matrix +
 * assign_add): cm[label, pred] += 1 for every pixel (rows = label, cols = prediction).
 *   cm [NC*NC] i64 accumulated in place (the caller zeroes it once).  Pairs outside [0,NC) are an
 *   error in TF; here they are counted in *dropped (i64, may be NULL) and otherwise ignored. */
int pcls_confusion_update(const int32_t* label, const int32_t* pred, int64_t n, int num_classes,
                          int64_t* cm, int64_t* dropped, pcls_stream stream);

/* test_step on the device, forward only (nets/SegmentationNetwork.py:118-131): ONE pass over the forward's outputs
 * accumulates the loss sums and the class-weighted confusion matrix.
 *   probs [n,NC] f32, label [n] i32, pred [n] i32 (NULL when cm_w is NULL), mask [n] u8 or NULL (= all valid),
 *   weight [n] f32 or NULL (= 1)
 *   loss_kind 0: none; 1: focal loss (:71-91) - loss_acc[0] += sum((1 - p)^gamma * -log(p) * weight * mask) with
 *             p = probs[label] + eps, loss_acc[1] += sum(mask); 2: Keras SparseCategoricalCrossentropy on probabilities
 *             (:49, :125) - loss_acc[0] += sum(-(log clip(p[label]) - log sum_c clip(p_c)) * weight), loss_acc[1] += n
 *             (clip to [1e-7, 1 - 1e-7]).  The caller divides (and applies CLS_LOSS_COEF).
 *   loss_acc [2] f64 accumulated in place; cm_w [NC*NC] f64 accumulated in place or NULL: cm_w[label, pred] += weight
 *   (tf.math.confusion_matrix(..., weights), :129); pairs outside [0,NC) are counted in *dropped (may be NULL).  NC <= 32. */
int pcls_validation_update(const float* probs, const int32_t* label, const int32_t* pred, const uint8_t* mask,
                           const float* weight, int64_t n, int num_classes, int loss_kind, double eps, double gamma,
                           double* loss_acc, double* cm_w, int64_t* dropped, pcls_stream stream);

/* Multi-GPU exchange step (no reference call site - the reference is single-device): sums the
 * per-GPU matrices in place with one ncclAllReduce(int64, sum) on `stream`.
 * The communicator helpers wrap the NCCL the process already has loaded (dlopen libnccl.so.2). */
#define PCLS_NCCL_UNIQUE_ID_BYTES 128
int pcls_comm_unique_id(char* h_id /* [128] out */);
int pcls_comm_init(void** comm, int nranks, const char* h_id, int rank);
int pcls_comm_destroy(void* comm);
int pcls_confusion_allreduce(int64_t* cm, int num_classes, void* comm, pcls_stream stream);

/* =====================================================================================
 * Network forward (SqueezeSegV2 / Darknet21 / Darknet53)
 * =====================================================================================
 * The Python model builders (pclsegmentation_b200/nets/*.py, mirroring the reference's
 * nets/SqueezeSegV2.py and nets/Darknet.py) describe the layer graph to a pcls_net op by op, passing
 * the raw Keras variables; the library folds BatchNorm (eps as given; Keras default 1e-3) into the
 * convolution, packs weights for the tensor-core kernels and plans the activation workspace.
 * pcls_net_forward then runs the whole graph for a batch: replaces model([lidar, mask])
 * (inference.py:75, eval.py:47) == SqueezeSegV2.call (nets/SqueezeSegV2.py:285-325) /
 * Darknet.call (nets/Darknet.py:279-314).
 *
 * Tensors are NHWC, 16-bit storage, identified by small integer ids.  Tensor 0 is the network
 * input: [B,H,W,8] = 6 input channels (5 normalised lidar channels + mask) + 2 zero pad channels. */

typedef struct pcls_net pcls_net;

enum { PCLS_F16 = 0, PCLS_BF16 = 1 };
enum { PCLS_ACT_NONE = 0, PCLS_ACT_RELU = 1, PCLS_ACT_LEAKY = 2 /* LeakyReLU(0.1) */ };
enum {
  PCLS_CONV = 0,          /* tf.keras.layers.Conv2D, padding SAME (VALID == SAME for 1x1), kernel [kh,kw,Cin,Cout] */
  PCLS_DECONV_1x4_S2 = 1  /* tf.keras.layers.Conv2DTranspose(kernel [1,4], strides [1,2], SAME), kernel [1,4,Cout,Cin] */
};

typedef struct pcls_conv_desc {
  int kind;               /* PCLS_CONV | PCLS_DECONV_1x4_S2 */
  int kh, kw;             /* 1x1, 3x3 (PCLS_CONV) or 1x4 (deconv) */
  int stride_w;           /* 1 or 2 (strides=[1,stride_w]; H is never strided in the reference) */
  int cin, cout;
  const float* h_kernel;  /* host, Keras layout (see kind) */
  const float* h_bias;    /* host [cout] or NULL (use_bias=False) */
  const float* h_bn_gamma; /* host [cout] x4 or all NULL (no BatchNormalization after the conv) */
  const float* h_bn_beta;
  const float* h_bn_mean;
  const float* h_bn_var;
  float bn_eps;
  int act;                /* activation applied after conv+bias+BN */
  int in_tensor;
  int out_tensor;         /* destination tensor; its channel count may exceed cout (tf.concat as a */
  int out_channel_offset; /* channel-offset write: SqueezeSegV2.py:127,199) */
  int residual0;          /* tensor ids added AFTER the activation (x += residual, Darknet.py:65,275; */
  int residual1;          /* tf.add skips, SqueezeSegV2.py:313-319), read at out_channel_offset; -1 = none */
  int out_is_logits;      /* 1: write float32 logits (conv14 / head), out_tensor must be a logits tensor */
} pcls_conv_desc;

/* precision: PCLS_F16 | PCLS_BF16 storage (fp32 accumulation always). */
int pcls_net_create(pcls_net** out, int H, int W, int precision, int max_batch);
void pcls_net_destroy(pcls_net* net);

/* Declares an activation tensor [B, H, width, channels]; returns its id (>= 1) or a negative status.
 * is_logits = 1 declares the float32 logits tensor [B,H,width,channels]. */
int pcls_net_tensor(pcls_net* net, int width, int channels, int is_logits);

int pcls_net_conv(pcls_net* net, const pcls_conv_desc* desc);

/* tf.nn.max_pool2d(ksize=3, strides=[1,2], padding='SAME') (SqueezeSegV2.py:295,301,305). */
int pcls_net_maxpool3x3_s2(pcls_net* net, int in_tensor, int out_tensor);

/* CAM.call (SqueezeSegV2.py:66-70): out = x * sigmoid(BN(1x1(relu(BN(1x1(maxpool7x7_SAME(x))))))).
 * sq_* : squeeze conv [1,1,C,C/r] (+bias) + BN; ex_* : excitation conv [1,1,C/r,C] (+bias) + BN. */
typedef struct pcls_cam_desc {
  int channels, reduced;
  const float *h_sq_kernel, *h_sq_bias, *h_sq_gamma, *h_sq_beta, *h_sq_mean, *h_sq_var;
  const float *h_ex_kernel, *h_ex_bias, *h_ex_gamma, *h_ex_beta, *h_ex_mean, *h_ex_var;
  float bn_eps;
  int in_tensor, out_tensor;
} pcls_cam_desc;
int pcls_net_cam(pcls_net* net, const pcls_cam_desc* desc);

/* Plans the workspace, uploads packed weights, builds TMA descriptors.  After this the op list is frozen. */
int pcls_net_finalize(pcls_net* net, int logits_tensor, int num_classes, int none_index);

/* Runs the graph on a batch.
 *   lidar    [B,H,W,channels] f32 (NULL with channels == 0: the input was staged in place, see pcls_net_input_buffers).
 *            channels == 6 and h_mean5 == NULL: the already normalised
 *            reference input (inference.py:56-62), channel 5 = mask.  channels == 5 or 6 with
 *            h_mean5/h_std5 given: RAW x,y,z,i,d(,label) - the input stage (inference.py:50-62) is
 *            fused into the load (mask = depth > 0).
 *   mask     [B,H,W] u8 (the reference's lidar_mask) or NULL = derive (channel 5 != 0, or depth > 0 for raw input)
 *   logits   [B,H,W,NC] f32 or NULL;  probs [B,H,W,NC] f32 or NULL;  preds [B,H,W] i32 (required)
 * B <= max_batch. */
int pcls_net_forward(pcls_net* net, const float* lidar, int channels, const uint8_t* mask,
                     const double* h_mean5, const double* h_std5, int B, float* logits, float* probs,
                     int32_t* preds, pcls_stream stream);

/* The same forward for a 16-bit host contract: `lidar16` is the normalised reference input (inference.py:56-62) already
 * in the net's storage type (IEEE half for PCLS_F16, bfloat16 for PCLS_BF16), [B,H,W,6] (5 channels + mask channel) or
 * [B,H,W,8] (tensor 0's own layout, channels 6-7 ignored).  The host ships 12 / 16 bytes per pixel instead of 24; the
 * results are bit-identical to pcls_net_forward on the float32 input these values were rounded from.
 *   mask  [B,H,W] u8 or NULL = derive (channel 5 != 0). */
int pcls_net_forward_in16(pcls_net* net, const void* lidar16, int channels, const uint8_t* mask, int B,
                          float* logits, float* probs, int32_t* preds, pcls_stream stream);

/* The net's input buffers, for producers that write the network input in place (pcls_project_resolve_net_input):
 * *input8 = tensor 0, [frames,H,W,8] 16-bit; *mask = [frames,H,W] u8; *frames = frames per pass (max_batch, or the micro
 * batch).  A forward over such a staged input is pcls_net_forward(net, NULL, 0, NULL, NULL, NULL, B <= frames, ...). */
int pcls_net_input_buffers(pcls_net* net, void** input8, uint8_t** mask, int* frames);

/* Debug / test access: copies activation tensor `tensor` of the last forward as float32 NHWC into
 * `out` ([B,H,width,channels] f32, device). */
int pcls_net_read_tensor(pcls_net* net, int tensor, int B, float* out, pcls_stream stream);

/* Per-op measurement for the roofline tables (bench.py, DESIGN.md): runs ONE forward like pcls_net_forward but
 * brackets every op with CUDA events on `stream` and returns the device time of each in h_ms (host, length
 * pcls_net_num_ops()).  Op 0 is the input kernel, the last op is the head.  Synchronises the stream. */
int pcls_net_num_ops(const pcls_net* net);
int pcls_net_profile_ops(pcls_net* net, const float* lidar, int channels, const uint8_t* mask,
                         const double* h_mean5, const double* h_std5, int B, float* logits, float* probs,
                         int32_t* preds, float* h_ms, pcls_stream stream);
/* Static description of op `i` for a batch of one frame: a short name (h_name, >= 64 bytes), which kernel
 * family runs it (0 = CUDA-core elementwise/direct, 1 = tcgen05 implicit GEMM), its algorithmic FLOPs and
 * its algorithmic bytes (external inputs + outputs at the storage width + weights), per frame. */
int pcls_net_op_info(const pcls_net* net, int i, char* h_name, int* family, int64_t* flops_per_frame,
                     int64_t* bytes_per_frame);

/* Introspection used by bench.py: number of kernel launches one forward enqueues, and workspace bytes. */
int pcls_net_launches_per_forward(const pcls_net* net);
int64_t pcls_net_workspace_bytes(const pcls_net* net);

/* Execution knobs (all CUDA; for A/B measurement and debugging):
 *   "conv_impl"  0 = tcgen05 implicit-GEMM where the shape allows (default), 1 = CUDA-core direct kernel
 *   "use_graph"  1 = replay the forward as a CUDA graph (default), 0 = plain launches
 *   "micro_batch" frames per pass through the graph (0 = whole batch)
 *   "fuse_head"  1 = softmax / argmax / mask in the epilogue of the final convolution (default), 0 = separate kernel
 *   "keep_tensors" (before finalize) 1 = no workspace reuse: every intermediate tensor of the last forward stays readable
 *                with pcls_net_read_tensor (per-layer parity tests); default 0 = liveness-planned arena
 *   "fuse_skip"  (before finalize) 1 = a 1x1 convolution of the network input with no activation whose only reader adds it
 *                as a skip after its ReLU (SqueezeSegV2's conv1_skip -> fire13 expand) is computed in that reader's epilogue
 *                and never written (default; off with keep_tensors or conv_impl = 1), 0 = its own launch and tensor
 * planning switches of the tcgen05 path, process-wide, to be set BEFORE pcls_net_finalize (all default 1):
 *   "tc_halo" (one 130-pixel tile serves three horizontal taps), "tc_resident" (weights stay in smem), "tc_group"
 *   (pixel-group view for 16 / 32-channel inputs), "tc_tma_store" (TMA-store epilogue), "tc_res_tma" (residual blocks
 *   TMA-loaded into the output staging buffers), "tc_split" (outer taps skip the expand1x1 half of merged Fire expands)
 *   "tc_nsplit" (N-split across CTAs with resident weight halves), "tc_head" (logits layer on its own kernel),
 *   "pad48" / "pair_s2" (before the first pcls_net_conv: 48-channel tensors stored with a 64-channel stride; 3x3 stride-2
 *   convolutions with 32 input channels on the pixel-pair view)
 * launch-time switches (any time; cached CUDA graphs are dropped):
 *   "tc_rtma"  bit 0: compile-time specialised residual kernel (one TMA-loaded skip tensor, TMA store, ReLU / LeakyReLU),
 *              bit 1: specialised plain kernel (no residual, TMA store); default 3, 0 = the generic kernel everywhere
 *              (a layer planned with a fused skip always runs its own specialised kernel)
 *   "cam_px"   pixels per thread of the CAM kernel: 0 = default (2), 1, 2
 * "tc_debug" (wait-cycle counters) needs a library built with PCLS_NVCC_FLAGS=-DPCLS_TC_DEBUG=1. */
int pcls_net_set_option(pcls_net* net, const char* name, int value);

#ifdef __cplusplus
}
#endif
#endif /* PCLSEG_H_ */
