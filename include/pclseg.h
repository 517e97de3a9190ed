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

/* Per-point labels from the range-image predictions (no reference call site: the reference stops at [H,W]
 * predictions, inference.py:78).  A k-NN vote in a search x search window of the range image, neighbours ranked by
 * range difference (the post-processing published with RangeNet++), so that a point that lost its pixel to a nearer
 * point does not simply take that point's label.
 *   preds        [B,H,W] i32   the forward's predictions, each in [0, num_classes)
 *   keys         [B,H,W] u64   winner keys left by pcls_project_scatter (either variant; ~0 = empty pixel)
 *   offsets      [B+1]  i64;  proj_x, proj_y [total] i32, unproj_range [total] f32 from the same scatter
 *   search       odd window size 1..9; 1 = plain back-projection (the label of the point's own pixel)
 *   k            1 <= k <= min(search*search, 32)
 *   h_window_weights  host f32 [search*search] (row-major, centre at search*search/2), finite and >= 0, or NULL = all 1
 *   cutoff       neighbours with weighted distance > cutoff do not vote; <= 0 = no cutoff
 *   ignore_class votes for this class are not counted; -1 = none
 *   pixel_scratch [B,H,W] u64 caller-provided when search > 1 (may be NULL when search == 1)
 *   point_labels [total] i32 out.  num_classes <= 32, 0 <= none_index < num_classes.
 * Rules (all deterministic): a dropped point (proj_x < 0) gets none_index.  Point i of scan b at pixel (r, c) with range
 * rho; window entry j = (dy+p)*search + (dx+p), p = (search-1)/2.  An entry outside the image (no column wrap-around) or
 * on an empty pixel is invalid.  A valid entry's range rho_j is unproj_range[offsets[b] + (key & 0xffffffff)] (the
 * centre entry uses rho itself) and its label preds[b, r+dy, c+dx].  d_j = |rho_j - rho| * w_j in float32 (separate
 * roundings).  The k valid entries with the smallest d_j are selected (ties: lower j; all of them if fewer than k); an
 * entry votes if d_j <= cutoff (or cutoff <= 0) and its label is not ignore_class.  The label is the class with the most
 * votes, ties to the lowest class; with no votes, the centre pixel's prediction. */
int pcls_point_labels(const int32_t* preds, const uint64_t* keys, const int64_t* offsets, int B, int H, int W,
                      int64_t total_points, const int32_t* proj_x, const int32_t* proj_y, const float* unproj_range,
                      int num_classes, int none_index, int search, int k, const float* h_window_weights,
                      float cutoff, int ignore_class, uint64_t* pixel_scratch, int32_t* point_labels,
                      pcls_stream stream);

/* Instance ids for thing-class points (no reference call site: the reference reads instance ids, SemLaserScan.set_label
 * inst = label >> 16, but never produces them): connected components in the range image.  The rules are this project's;
 * bit parity with any published clustering code is not claimed.
 *   points       [total,4] f32 (16-byte aligned), keys [B,H,W] u64, offsets, proj_x, proj_y: pcls_project_scatter's
 *                (either variant: the key's low word is the winner's local index)
 *   point_labels [total] i32 L, e.g. from pcls_point_labels;  thing_mask: bit c set = class c is a thing class
 *                (1 <= num_classes <= 32, no bit at or above num_classes; labels outside [0, num_classes) are never things)
 *   scratch      caller-provided, 16-byte aligned, pcls_point_instances_scratch_bytes(B, H, W) bytes
 *   instances    [total] i32 out;  instance_counts [B] i32 out: the number of ids in each scan
 * Rules, per scan b:
 *   1. A node is a pixel (r, c) whose winner point i (offsets[b] + low word of the key) has L[i] in the thing set.
 *   2. Nodes u and v are joined when |r_u - r_v| <= ry; the column distance is <= rx (modulo W with wrap = 1, because a
 *      360-degree scan's columns 0 and W-1 are neighbours; no wrap-around with wrap = 0); L is equal at the two nodes; and
 *      d^2 <= tau^2, d^2 = (dx*dx + dy*dy) + dz*dz in float32 with separate roundings over the two winners' x, y, z,
 *      tau^2 = fl32(tau * tau).
 *   3. Components are the connected components of that graph.
 *   4. A node's winner belongs to the node's component.  A non-winner point j whose pixel is a node belongs to that
 *      component when L[j] equals the winner's label and d^2(j, winner) <= tau^2.  Every other point (stuff classes,
 *      dropped points with proj_x < 0, occluded points that fail the test) belongs to no component.
 *   5. A component's size is the number of points that belong to it.  Components with size >= min_points are numbered
 *      1, 2, ... per scan in increasing order of their smallest pixel index r*W + c; every other point gets 0.
 *   6. 0 <= ry <= 4, 0 <= rx <= 8, ry + rx > 0, 2 rx < W when wrapping, tau finite and > 0, min_points >= 1,
 *      B*H*W < 2^31; otherwise PCLS_ERR_INVALID.
 * The output is fully determined: the same bits on every run, whatever order the atomics land in.
 * pcls_point_instances_scratch_bytes returns the bytes (24 per pixel), or PCLS_ERR_INVALID for bad sizes. */
int64_t pcls_point_instances_scratch_bytes(int B, int H, int W);
int pcls_point_instances(const float* points, const uint64_t* keys, const int64_t* offsets, int B, int H, int W,
                         int64_t total_points, const int32_t* proj_x, const int32_t* proj_y,
                         const int32_t* point_labels, int num_classes, uint32_t thing_mask, int ry, int rx, int wrap,
                         float tau, int min_points, void* scratch, int32_t* instances, int32_t* instance_counts,
                         pcls_stream stream);

/* Test-time augmentation (no reference call site: the configs train with RANDOM_FLIPPING and SHIFT_LEFT_RIGHT, the
 * reference infers on one view).  The rules are this project's; parity with the reference's training-time flip / shift
 * code is not claimed.
 *   A view is (flip, shift), flip in {0, 1}, 0 <= shift < W: a permutation of the columns of a raw range image plus a
 *   rigid transform of its points.  For source pixel (h, w):
 *     mirror (flip = 1): column w -> W-1-w and y -> -y (the scan mirrored across the x axis: yaw = -atan2(y, x) puts
 *       column p at W - p, up to points exactly on a column boundary);
 *     roll by shift: column w -> (w + shift) mod W, and (x, y) rotated about z by alpha = -2 pi shift / W:
 *       x' = c x - s y, y' = s x + c y with c = h_cos[t], s = h_sin[t] (the sensor turned by `shift` columns; the
 *       column grows with yaw).  c and s are computed on the host in float64; for shift a multiple of W/4 they are exactly
 *       0 and +-1, so the half turn is x -> -x, y -> -y.  With shift = 0 the points are not rotated at all.
 *     The mirror comes first, then the roll.  z, remission and range are unchanged; the mask is range > 0.
 *   Frame order is view-major: view t of frame b is frame t*B + b.
 * pcls_tta_views: raw [B,H,W,channels] f32 (channels 5 or 6; the label channel is ignored) -> for every view the
 *   network input `input8` [n_views*B,H,W,8] 16-bit (precision PCLS_F16 | PCLS_BF16) and `mask` [n_views*B,H,W] u8, e.g.
 *   the net's own buffers (pcls_net_input_buffers).  Per view pixel: the rotation in float64 from the float32 inputs
 *   with separate roundings (c*x and s*y rounded, then their difference / sum), then the input stage of
 *   pcls_net_forward's raw path, (float)((v - mean) / std) in float64 rounded to float32 and then to 16 bits; empty
 *   pixels are zeros, channel 5 is the mask, channels 6-7 are zero.  View (0, 0) is bit-identical to the tensor 0 that
 *   pcls_net_forward makes of raw input and to pcls_project_resolve_net_input's.
 * pcls_tta_merge: probs [n_views*B,H,W,num_classes] f32 (the forward over the views), mask [n_views*B,H,W] u8 (the views'
 *   masks) -> per output pixel (b, h, w) of the source image, with q_t the pixel of view t that (b, h, w) maps to:
 *   acc = probs[q_0]; acc = acc + probs[q_t] for t = 1 .. n_views-1 in float32 (round to nearest); mean = acc / n_views
 *   (T = 1 returns probs[q_0] unchanged); out_preds [B,H,W] i32 = argmax of the means (first index on ties, the head's
 *   rule), none_index where mask[q_0] == 0; out_probs [B,H,W,num_classes] f32 = the means, or NULL.
 * Both calls check before any launch: 1 <= n_views <= PCLS_TTA_MAX_VIEWS, flips 0 / 1, shifts in [0, W), no view twice,
 * finite h_cos / h_sin, channels 5 / 6, 1 <= num_classes <= 32, 0 <= none_index < num_classes, and the pointers the call
 * needs; otherwise PCLS_ERR_INVALID. */
#define PCLS_TTA_MAX_VIEWS 8
int pcls_tta_views(const float* raw, int channels, int B, int H, int W, const double* h_mean5, const double* h_std5,
                   int n_views, const int* h_flip, const int* h_shift, const double* h_cos, const double* h_sin,
                   int precision, void* input8, uint8_t* mask, pcls_stream stream);
int pcls_tta_merge(const float* probs, const uint8_t* mask, int B, int H, int W, int num_classes, int none_index,
                   int n_views, const int* h_flip, const int* h_shift, float* out_probs, int32_t* out_preds,
                   pcls_stream stream);

/* Calibrated confidence (no reference call site: the reference reduces the softmax to an argmax).  Post-hoc temperature
 * scaling (Guo et al., "On Calibration of Modern Neural Networks", ICML 2017): one scalar T, probabilities softmax(z / T).
 * The argmax does not depend on T.  The host passes a = 1/T, computed in float64 and rounded once to float32.
 * All four calls check every argument before any launch (1 <= num_classes <= 32, the pointers the call needs; otherwise
 * PCLS_ERR_INVALID with a pcls_last_error message); n == 0 is a no-op.
 * pcls_confidence: exactly one of logits / probs [n,NC] f32 is non-NULL; a finite and > 0, and a == 1 in probs mode.
 *   Logits mode: v_c = z_c * a rounded to float32, then the head's softmax (pcls_head's arithmetic: at a = 1 out_probs is
 *   bit-identical to pcls_head's probabilities; the fused conv_head path uses ex2.approx and is not).  Probs mode: p = probs.
 *   out_conf [n] f32 = max_c p_c; out_entropy [n] f32 = (-sum_c p_c * logf(p_c)) over the classes with p_c > 0, summed in
 *   class order in float32 (products and sums rounded one at a time), divided by logf(NC); 0 when NC = 1.  Where
 *   mask[i] == 0 (mask [n] u8, NULL = all valid) conf and entropy are 0.  out_probs [n,NC] f32 is written for every pixel,
 *   as the head does.  Each output may be NULL, at least one must be given.
 * pcls_temperature_nll: the NLL of softmax(z * a_t) for n_temps (1..64) inverse temperatures h_inv_temps (host f32, each
 *   finite and > 0) in one pass over logits [n,NC] f32.  A pixel counts when 0 <= label < NC and label != ignore_index
 *   (label [n] i32).  Per counted pixel and t, in float32 with separate roundings: s_c = z_c * a_t, m = max_c s_c,
 *   e = sum_c expf(s_c - m) in class order, term = (logf(e) + m) - s_label.  nll_acc [n_temps] f64 += term (float64 sums,
 *   order unspecified), counted [1] i64 += 1 per counted pixel; both accumulated in place.
 * pcls_reliability_update: the reliability histogram of n_bins (1..64) equal bins of [0, 1].  An element counts when
 *   0 <= label < NC, label != ignore_index and 0 <= pred < NC (conf [n] f32, pred / label [n] i32).  Its bin is
 *   b = min((int)(conf * (float)n_bins), n_bins - 1) with the product rounded to float32 (clamped at 0 below);
 *   bin_count[b] (i64) += 1, bin_correct[b] (i64) += (pred == label), bin_conf[b] (f64) += conf, accumulated in place.
 *   The host computes ECE = sum_b |bin_correct_b - bin_conf_b| / N, MCE over the non-empty bins, accuracy and mean
 *   confidence from these sums.
 * pcls_point_confidence: per point i of scan b (offsets [B+1] i64, proj_x / proj_y [total] i32 of pcls_project_scatter,
 *   point_labels [total] i32, probs [B,H,W,NC] f32): out_conf[i] = probs[b, proj_y[i], proj_x[i], point_labels[i]], the
 *   probability the point's own pixel gives the label the point got; 0 for a dropped point (proj_x < 0) or a label
 *   outside [0, NC).  An exact gather. */
int pcls_confidence(const float* logits, const float* probs, const uint8_t* mask, int64_t n, int num_classes,
                    float inv_temperature, float* out_probs, float* out_conf, float* out_entropy, pcls_stream stream);
int pcls_temperature_nll(const float* logits, const int32_t* label, int64_t n, int num_classes, int ignore_index,
                         int n_temps, const float* h_inv_temps, double* nll_acc, int64_t* counted, pcls_stream stream);
int pcls_reliability_update(const float* conf, const int32_t* pred, const int32_t* label, int64_t n, int num_classes,
                            int ignore_index, int n_bins, int64_t* bin_count, int64_t* bin_correct, double* bin_conf,
                            pcls_stream stream);
int pcls_point_confidence(const float* probs, const int64_t* offsets, int B, int H, int W, int64_t total,
                          const int32_t* proj_x, const int32_t* proj_y, const int32_t* point_labels, int num_classes,
                          float* out_conf, pcls_stream stream);

/* Monte-Carlo dropout (Gal & Ghahramani, ICML 2016; Kendall et al., Bayesian SegNet, 2015): T forward passes of a
 * stochastic net whose Dropout layers are active; the mean probabilities, the predictive entropy and the mutual
 * information between prediction and weights.  No reference call site: the reference's Dropout layers act in training only.
 * Dropout site: one Dropout call of the model, numbered in trace order (SqueezeSegV2: site 0 = fire13 + conv1_skip, 64
 * channels at full width; Darknet: sites 0-4 = the outputs of enc1 .. enc5, site 5 = the input of head).  A site modifies
 * its tensor IN PLACE: every later reader sees the dropped tensor.
 * Mask: element e = (h * W_t + w) * C + c of frame f's tensor (C a multiple of 8), pass t (0 <= t < 65536), site k
 *   (0 <= k < 65536), f the GLOBAL frame id = frame_base + the frame's index in the forward call (micro-batch passes
 *   counted).  Philox4x32-10 (Salmon et al., SC 2011) with counter (g, k | t << 16, lo32(f), hi32(f)), g = e / 8, and key
 *   (lo32(seed), hi32(seed)); output word i (0..3) gives u (16 bits) to two elements: its low half to element 8g + 2i,
 *   its high half to element 8g + 2i + 1.  thr = floor(rate * 65536 + 0.5) in float64 (0 <= rate, thr < 65536, else
 *   PCLS_ERR_INVALID); the element is kept iff u >= thr, and then becomes round16_rn(fl32(x) * scale) with
 *   scale = (float)(65536.0 / (65536 - thr)) (computed in float64, rounded once, the product rounded to float32); a
 *   dropped element becomes the bit pattern 0.  At rate 0 the tensor is bit-for-bit unchanged.  The mask of a frame
 *   depends only on (seed, global frame id, pass, site): not on the batch, the micro batch, graph replay or the number of
 *   GPUs.  Parity with TensorFlow's dropout RNG is not claimed.
 * pcls_net_dropout (before pcls_net_finalize): appends the in-place dropout of activation `tensor` as site `site` at
 *   `rate` to the op list.  Refused (PCLS_ERR_INVALID): the network input or a logits tensor, a tensor no earlier op
 *   writes, channels not a multiple of 8 or a pixel stride other than the channel count (the 48 -> 64 padded tensors), a
 *   site used twice, an invalid rate; pcls_net_finalize refuses a site tensor the planner fuses away.  The op is listed
 *   by pcls_net_num_ops / pcls_net_op_info / pcls_net_profile_ops like any other.
 * pcls_net_set_dropout: writes the net's device-side (seed, frame_base, pass) with a one-thread kernel on `stream`,
 *   outside the forward's CUDA graph: the dropout kernels read it, so one captured graph serves every pass and batch.
 *   Needs a finalized net with at least one dropout op and 0 <= pass < 65536.  The state starts as (0, 0, 0).
 * pcls_mc_accumulate: probs [n,NC] f32 of pass `pass`; h_t = the normalised entropy of probs as pcls_confidence computes
 *   it.  pass 0: acc_probs [n,NC] f32 = probs, acc_entropy [n] f64 = (double)h_0; pass > 0: acc_probs = fl32(acc_probs +
 *   probs) (round to nearest), acc_entropy += (double)h_t.  Passes are accumulated in the order of the calls.
 * pcls_mc_finalize over n_passes = T (1 .. 65536): mean = acc_probs / T (__fdiv_rn; T = 1 leaves acc_probs unchanged);
 *   out_preds [n] i32 = argmax of mean (first index on ties, the head's rule), none_index where mask == 0 (mask [n] u8,
 *   NULL = all valid); out_conf [n] f32 = max mean; out_entropy [n] f32 = H, the normalised entropy of mean by the same
 *   rule as h_t; out_mi [n] f32 = max(0, fl32(H - EH)) with EH = (float)(acc_entropy / T); conf / H / MI are 0 where
 *   mask == 0; out_probs [n,NC] f32 = mean, written for every pixel as the head does.  Each output may be NULL, at least
 *   one must be given.  At rate 0 with T = 1 or 2, mean and preds are the plain forward's bits and MI is 0; from T = 3
 *   on the running float32 sum rounds (3p is not exact), so the mean is within a few ulp of the plain probabilities.
 * Both calls check every argument before any launch (1 <= num_classes <= 32, 0 <= none_index < num_classes, the pointers
 * the call needs); n == 0 is a no-op.  pcls_net_dropout / pcls_net_set_dropout are declared with the net below. */
int pcls_mc_accumulate(const float* probs, int64_t n, int num_classes, int pass, float* acc_probs, double* acc_entropy,
                       pcls_stream stream);
int pcls_mc_finalize(const float* acc_probs, const double* acc_entropy, const uint8_t* mask, int64_t n, int num_classes,
                     int none_index, int n_passes, float* out_probs, int32_t* out_preds, float* out_conf,
                     float* out_entropy, float* out_mi, pcls_stream stream);

/* Semantic map fusion (no reference call site: the reference labels each scan on its own).  The point labels of a
 * pose-registered sequence are voted into a voxel hash map, and points are relabelled from it.  The rules are this
 * project's; parity with SuMa++ or any other mapping code is not claimed.
 * Voxel of a point: point i of scan b has float32 (x, y, z) from points [total,4] f32 (16-byte aligned) and offsets [B+1]
 *   i64.  poses [B,12] f64 is a DEVICE array: the 3x4 row-major lidar-to-world transform (R | t) of each scan.  World
 *   coordinate w_k = ((R_k0*x + R_k1*y) + R_k2*z) + t_k in float64, every product and sum rounded on its own (no FMA
 *   contraction).  v_k = floor(w_k / s), s = voxel_size, IEEE float64 division.  A point has no voxel when a w_k is not
 *   finite or a v_k is outside [-2^20, 2^20).  Key = ((vx + 2^20) << 42) | ((vy + 2^20) << 21) | (vz + 2^20) as u64,
 *   always below 2^63, so ~0 marks an empty slot.
 * Table: table_keys [capacity] u64 and table_counts [capacity, NC] u32, capacity a power of two, 1 <= NC <= 32.  An empty
 *   table is all keys ~0 and all counts 0.  state [2] i64: state[0] = occupied slots; state[1] = points (or, when
 *   growing, keys) that found no free slot within `capacity` probes - 0 while the load stays at most 1/2, there so that
 *   misuse cannot hang a kernel.  The hash and the probe sequence are internal; slot placement depends on the order of
 *   atomics, but the set of (key, counts), the query results and an export sorted by key are the same bits on every run.
 * pcls_semantic_map_vote: a point votes when it has a voxel, 0 <= labels[i] < NC, labels[i] != ignore_class, and
 *   r2 >= min_range^2 and (max_range <= 0 or r2 <= max_range^2), r2 = (x*x + y*y) + z*z in float64 with separate roundings
 *   in the sensor frame, the squared limits computed in float64.  A vote inserts the key if it is new (state[0] += 1) and
 *   then adds 1 to table_counts[slot, label].
 * pcls_semantic_map_grow: initialises the new table itself (keys ~0, counts 0) and reinserts every occupied slot of the
 *   old one with its row of counts; state[0] is unchanged.  new_capacity must be a power of two at least twice state[0]
 *   (the host may pass a bound it holds instead of reading state[0]).  The tables must not overlap.
 * pcls_semantic_map_query: per point, out_labels[i] = labels_in[i] when it is a class of keep_mask (bit c = class c);
 *   otherwise, when its voxel is in the table with at least min_votes (>= 1) votes in total, the argmax of the voxel's
 *   counts (ties to the lowest class); otherwise labels_in[i].  The range limits do not apply: a far point, or one the
 *   projection dropped, takes the label of a voxel that nearer scans established.
 * Every call checks before any launch: 1 <= NC <= 32; ignore_class -1 or in [0, NC); no keep_mask bit at or above NC;
 * voxel_size finite and > 0; finite range limits with 0 <= min_range and (max_range <= 0 or max_range >= min_range);
 * capacities powers of two; total < 2^31; the pointers the call needs.  Otherwise PCLS_ERR_INVALID.  Pose entries live
 * on the device and are not checked here (semantic_map.SemanticMap checks them).  total == 0 is a no-op. */
int pcls_semantic_map_vote(const float* points, const int64_t* offsets, int B, int64_t total, const double* poses,
                           double voxel_size, double min_range, double max_range, const int32_t* labels,
                           int num_classes, int ignore_class, uint64_t* table_keys, uint32_t* table_counts,
                           int64_t capacity, int64_t* state, pcls_stream stream);
int pcls_semantic_map_grow(const uint64_t* old_keys, const uint32_t* old_counts, int64_t old_capacity, int num_classes,
                           uint64_t* new_keys, uint32_t* new_counts, int64_t new_capacity, int64_t* state,
                           pcls_stream stream);
int pcls_semantic_map_query(const float* points, const int64_t* offsets, int B, int64_t total, const double* poses,
                            double voxel_size, const int32_t* labels_in, int num_classes, uint32_t keep_mask,
                            int min_votes, const uint64_t* table_keys, const uint32_t* table_counts, int64_t capacity,
                            int32_t* out_labels, pcls_stream stream);

/* Per-point ground truth for point-wise evaluation: out[i] = lut[labels[i] & 0xFFFF], ids >= lut_len -> 0,
 * lut NULL -> the raw semantic id (the same rule pcls_project_resolve applies per pixel). */
int pcls_map_labels(const uint32_t* labels, int64_t n, const int32_t* label_lut, int lut_len, int32_t* out,
                    pcls_stream stream);

/* Per-frame statistics of range images [B,H,W,channels] (x, y, z, remission, range[, label]): the moments a config's
 * INPUT_MEAN / INPUT_STD come from, channel ranges, occupancy and class counts (the reference computes them offline with
 * numpy, preprocessing/inspect_training_data.py; the rules below are this project's, bit parity with its RunningStd is
 * not claimed).
 *   frames       dtype 0 = float32, 1 = float64 (the converters' .npy files, read without narrowing)
 *   channels     5 or 6;  h_shift5 host doubles (s_c) or NULL (= 0), finite
 *   frame_sums   [B,5,4] f64 OUT, per frame and channel: sum(d), sum(d*d), min(x), max(x), d = x - s_c,
 *                over the frame's VALID pixels (valid = range channel > 0 on the stored value; NaN is invalid).  A NaN
 *                value at a valid pixel enters the sums but not min / max.  A frame with no valid pixel gets sums of 0,
 *                min = +inf, max = -inf.  The summation order depends only on H, W and channels: a frame's row is the
 *                same bits whatever B is and wherever the frame sits in the batch.
 *   frame_valid  [B] i64 OUT: valid pixels per frame
 *   row_valid [H], col_valid [W], class_pixels [num_classes], dropped [1]: i64, ACCUMULATED, each may be NULL;
 *                class_pixels counts the label channel at valid pixels, truncated toward zero like pcls_input_stage's
 *                (int32_t) cast; a label that is not finite or not in [0, num_classes) increments *dropped
 *                (class_pixels / dropped need channels == 6 and 1 <= num_classes <= 32).  H, W <= 16384. */
int pcls_dataset_stats(const void* frames, int dtype, int channels, int B, int H, int W, const double* h_shift5,
                       int num_classes, double* frame_sums, int64_t* frame_valid, int64_t* row_valid,
                       int64_t* col_valid, int64_t* class_pixels, int64_t* dropped, pcls_stream stream);

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
 *           (label and weight require channels == 6).
 * Label rule at valid pixels (the label channel is a float): like parse_sample, the weight compares the FLOAT label with
 * each class id, so weight = CLS_LOSS_WEIGHT[l] only if the label equals the integer l exactly (-0.0 counts as 0);
 * fractional (2.5), NaN, +-inf, negative and >= num_classes labels get 0.  label = the float truncated toward zero,
 * saturated to the int32 range, NaN -> 0 (numpy's astype leaves NaN / out-of-range to the host; integer labels in range
 * are the same either way). */
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

/* Adds a convolution.  Into a 16-bit (non-logits) tensor, out_channel_offset and cout must be multiples of 8, like the
 * channel count of every 16-bit tensor: outputs are written as whole 8-channel vectors.  Otherwise PCLS_ERR_INVALID. */
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
 *   mask     [B,H,W] u8 (the reference's lidar_mask) or NULL = derive: channel 5 != +-0 after its rounding to the
 *            storage type (so a float32 channel 5 that rounds to a 16-bit zero is an empty pixel, NaN a valid one), or
 *            depth > 0 for raw input.  For raw input a given mask sets only which pixels are valid (the head's
 *            none_index); tensor 0's channel 5 and the zeroed channels still follow depth > 0.
 *   logits   [B,H,W,NC] f32 or NULL;  probs [B,H,W,NC] f32 or NULL;  preds [B,H,W] i32 (required)
 * B <= max_batch. */
int pcls_net_forward(pcls_net* net, const float* lidar, int channels, const uint8_t* mask,
                     const double* h_mean5, const double* h_std5, int B, float* logits, float* probs,
                     int32_t* preds, pcls_stream stream);

/* The same forward for a 16-bit host contract: `lidar16` is the normalised reference input (inference.py:56-62) already
 * in the net's storage type (IEEE half for PCLS_F16, bfloat16 for PCLS_BF16), [B,H,W,6] (5 channels + mask channel) or
 * [B,H,W,8] (tensor 0's own layout, channels 6-7 ignored).  The host ships 12 / 16 bytes per pixel instead of 24; the
 * results are bit-identical to pcls_net_forward on the float32 input these values were rounded from.
 *   mask  [B,H,W] u8 or NULL = derive (channel 5 != +-0; NaN is valid). */
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
 *   "fuse_up"    (before finalize) 1 = each FireDeconv squeeze 1x1 runs inside the transposed convolution behind it
 *                (default), 0 = two launches
 *   "fuse_pool"  (before finalize) 1 = each 3x3 / stride-2 max-pool runs inside the 1x1 convolution that reads it
 *                (default), 0 = its own launch and tensor
 *   "tc_debug"   1 = per-role wait-cycle counters of the tcgen05 kernel, printed per convolution by pcls_net_profile_ops;
 *                needs a library built with PCLS_NVCC_FLAGS=-DPCLS_TC_DEBUG=1
 * Any other name fails with PCLS_ERR_INVALID. */
int pcls_net_set_option(pcls_net* net, const char* name, int value);

/* MC dropout ops of a stochastic net (the rules are stated with pcls_mc_accumulate above). */
int pcls_net_dropout(pcls_net* net, int tensor, int site, double rate);
int pcls_net_set_dropout(pcls_net* net, uint64_t seed, uint64_t frame_base, int pass, pcls_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* PCLSEG_H_ */
