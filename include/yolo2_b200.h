/*
 * yolo2_b200.h -- C ABI of libyolo2_b200.so: the B200 (sm_100a) kernels behind the detection
 * hot path of wenxichen/tensorflow_yolo2 (Darknet19 forward, grid/region decode, NMS, YOLO loss).
 *
 * The reference has NO native interface (it is pure Python over TensorFlow 1.x); the "FFI" a
 * maintainer binds is therefore the set of TF-op call sites on the path.  Each entry point below
 * names the reference call site (file:line under the reference repo's src/) it replaces.  The
 * Python stub that binds these (ctypes) is shown in INTEGRATION.md and lives in
 * tensorflow_yolo2_b200/_lib.py.
 *
 * Conventions
 *   - extern "C"; plain pointers and sizes; no torch / C++ types in any signature.
 *   - All data pointers are DEVICE pointers owned by the caller unless the name says `host`.
 *   - Every function returns int: 0 = OK, <0 = bad argument (Y2_ERR_*), >0 = cudaError_t.
 *     y2_last_error() returns a thread-local message for the last failure.
 *   - No allocation and no host synchronisation inside (exception: y2_*_host helpers, which say
 *     so).  Work is enqueued on `stream` (a cudaStream_t passed as void*).
 *   - Tensors are NHWC; "rows" M = N*H*W pixels.  bf16 = __nv_bfloat16 bits.
 */
#ifndef YOLO2_B200_H_
#define YOLO2_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Y2_OK 0
#define Y2_ERR_BAD_ARG (-1)
#define Y2_ERR_UNSUPPORTED (-2)
#define Y2_ERR_WORKSPACE (-3)
#define Y2_ERR_DRIVER (-4)

typedef void* y2_stream_t; /* cudaStream_t */

/* ---- library ------------------------------------------------------------------------------ */
int y2_version(void);
const char* y2_last_error(void);
/* Number of kernels this library has launched from the calling process since load (all threads).
 * bench.py reports the delta over the timed region as "gpu_launches". */
unsigned long long y2_launch_count(void);
/* The Y2_* environment switches (reference paths for tests and tools, INTEGRATION.md section 5) are read once per process;
   this re-reads them. */
int y2_reload_env(void);

/* ---- a10: input preprocessing ------------------------------------------------------------
 * pascal_detect_darknet.py:36-37, img_dataset/pascal_voc.py:62-64:  x = (u8 / 255.0) * 2.0 - 1.0
 * on an already-resized BGR image.  out_dtype 0: float32 [N,H,W,3];  1: bf16 [N,H,W,8] with
 * channels 3..7 zero (the layout the first tensor-core conv consumes). */
int y2_preprocess_u8(const uint8_t* img, void* out, int N, int H, int W, int out_dtype, y2_stream_t stream);
/* cv2.resize(image, (dst_w, dst_h)) of pascal_detect_darknet.py:35 / img_dataset/pascal_voc.py:61 for an 8-bit 3-channel
 * image (default INTER_LINEAR), BIT-EXACT: OpenCV's fixed-point algorithm (2048-scaled short coefficients, clamped columns
 * with zeroed weights, clamped rows with kept weights, ((b * (R >> 4)) >> 16) vertical pass, + 2 >> 2; exact 2x down-scale ->
 * 2x2 area mean).  src uint8 [src_h, src_w, 3] (device), dst uint8 [dst_h, dst_w, 3] -- typically one row of the engine's
 * uint8 input batch, so the host never touches pixels after the JPEG decode. */
int y2_resize_bilinear_u8(const uint8_t* src, int src_h, int src_w, uint8_t* dst, int dst_h, int dst_w, y2_stream_t stream);
/* float32 [N,H,W,3] (already normalised, what the reference feeds sess.run) -> bf16 [N,H,W,8] */
int y2_pad_cast_f32_to_bf16c8(const float* x, void* out, int N, int H, int W, y2_stream_t stream);

/* ---- a1: convolution, exact float32 path ---------------------------------------------------
 * yolo2_nets/darknet.py:20-21 (tf.nn.conv2d SAME stride 1) + :35 (+ bias).
 * x [N,H,W,Cin] f32, w HWIO [k,k,Cin,Cout] f32 (the TF variable layout), y [N,H,W,Cout] f32.
 * FFMA kernel, fp32 accumulate: the "1e-5" path of the spec and the GPU cross-check of the
 * tensor-core kernel.  ksize in {1,3}. */
int y2_conv_fwd_f32(const float* x, const float* w_hwio, const float* bias, float* y,
                    int N, int H, int W, int Cin, int Cout, int ksize, y2_stream_t stream);

/* ---- a1+a2+a3 fused: convolution on tcgen05 tensor cores ----------------------------------
 * Same call sites as above plus darknet.py:42-45 (BN as per-channel scale/shift, leaky ReLU) and
 * :24-25 (2x2 max-pool) in the epilogue.  Implicit GEMM: A = activations via TMA (im2col or
 * tiled box mode) into swizzled smem, B = packed weights via TMA, D in TMEM, bf16 x bf16 -> fp32.
 *
 *   x        bf16 [N,H,W,Cin_p]    Cin_p = y2_conv_cin_padded(Cin)  (3 -> 8, else Cin)
 *   w_packed bf16 [Cout_p][k*k][Cin_p]  from y2_pack_weights_bf16  (Cout_p = Cout rounded up to 16,
 *            K padded with zero columns as y2_conv_packed_weight_elems says)
 *   epilogue v = acc * scale[c] + shift[c];  if LEAKY: v = max(v, alpha*v);  if POOL2: 2x2 max
 *   y        bf16 [N,Ho,Wo,Cout] (ldy = Cout)   or, with OUT_F32, float32 rows of stride ldy
 */
#define Y2_CONV_LEAKY 1
#define Y2_CONV_POOL2 2
#define Y2_CONV_OUT_F32 4
/* "bf16x3" precision mode (the 1e-3 detections bar of the spec; a single bf16 rounding per operand is ~1e-2 after 22
 * layers).  Every value v travels as TWO bf16 numbers hi = bf16(v), lo = bf16(v - hi) (16 mantissa bits together) and a
 * product a*w is evaluated as a_hi*w_hi + a_lo*w_hi + a_hi*w_lo -- three tcgen05.mma per K step into the same fp32
 * accumulator (the dropped a_lo*w_lo term is 2^-18 relative).
 *   IN_SPLIT   x is bf16 [N,H,W,2*Cin] = [hi(Cin) | lo(Cin)] per pixel and w_packed comes from
 *              y2_pack_weights_bf16_split (K per tap = 3*Cin: [w_hi | w_hi | w_lo], meeting x's [hi | lo | hi]).
 *              Cin must be a multiple of 32.
 *   OUT_SPLIT  the bf16 output row holds hi at columns [0, Cout) and lo at [lo_off, lo_off + Cout); ldy >= lo_off + Cout
 *              (lo_off = 0 means Cout: a dense [N,Ho,Wo,2*Cout] tensor).  Ignored with OUT_F32. */
#define Y2_CONV_IN_SPLIT 8
#define Y2_CONV_OUT_SPLIT 16
typedef struct y2_conv_params {
  const void* x;
  const void* w_packed;
  const float* scale; /* [Cout] or NULL (=1) */
  const float* shift; /* [Cout] or NULL (=0) */
  void* y;
  int N, H, W, Cin, Cout, ksize;
  int flags;
  float alpha;
  int ldy;      /* output row stride in elements; 0 -> Cout */
  int lo_off;   /* OUT_SPLIT: column of the lo half (0 -> Cout); must be 0 otherwise */
} y2_conv_params;
int y2_conv_cin_padded(int Cin);
size_t y2_conv_packed_weight_elems(int ksize, int Cin, int Cout);
int y2_pack_weights_bf16(const float* w_hwio, void* w_packed, int ksize, int Cin, int Cout, y2_stream_t stream);
/* IN_SPLIT operand: [Cout_p][k*k][3*Cin] bf16 = per tap [w_hi | w_hi | w_lo]; y2_conv_packed_weight_split_elems elements. */
size_t y2_conv_packed_weight_split_elems(int ksize, int Cin, int Cout);
int y2_pack_weights_bf16_split(const float* w_hwio, void* w_packed, int ksize, int Cin, int Cout, y2_stream_t stream);
int y2_conv_fwd_bf16(const y2_conv_params* p, y2_stream_t stream);

/* Scratch for the stream-K variant of y2_conv_fwd_bf16 (256x256 tiles whose K range is split between two CTAs: the
 * partial accumulators travel through this buffer).  Register a device buffer of y2_conv_workspace_bytes() bytes
 * (256-byte aligned) per calling thread; convolutions issued concurrently on different streams need different
 * buffers (the Python front end keeps one per (device, stream) and one per engine / trainer).  The first 4096 bytes
 * (hand-over flags) must be ZERO when the buffer is registered; every launch leaves them zero again.  Without a
 * workspace (or with NULL) every layer runs on the 128-row-tile kernel -- same results up to the float32 summation
 * order. */
size_t y2_conv_workspace_bytes(void);
int y2_conv_set_workspace(void* workspace, size_t bytes);

/* ---- a10+a1+a2+a3 fused for the FIRST layer (inference-mode BN): uint8 image -> pooled bf16 activation ---------
 * pascal_voc.py:62-64 (x/255*2-1) + darknet.py:150-151 (conv 3x3 3->32, +bias, BN, leaky, 2x2 max-pool) in one
 * kernel; the padded bf16 input is never materialised.  img uint8 [N,H,W,3] (H % 32 == 0, W % 16 == 0, 16-byte
 * aligned); w_packed from y2_pack_weights_conv1_u8 (the BN scale is folded INTO the bf16 weights because the kernel
 * pools before the affine/leaky step; `scale` NULL = 1); shift [32] = beta + (bias - mean) * scale;
 * y bf16 [N,H/2,W/2,32] = maxpool(leaky(conv * scale + shift)).  Cout is fixed at 32 (Darknet19). */
size_t y2_conv1_u8_packed_weight_elems(void);
int y2_pack_weights_conv1_u8(const float* w_hwio, const float* scale, void* w_packed, y2_stream_t stream);
int y2_conv1_u8_pool_fwd(const uint8_t* img, const void* w_packed, const float* shift, void* y, int N, int H, int W,
                         float alpha, y2_stream_t stream);
/* bf16x3 variant of the same layer: the raw bytes enter the MMA as exact bf16 integers plus a "ones" channel (1 inside
 * the image, 0 in the SAME-padding halo); x = v*2/255 - 1 is folded into the weights, which are a hi + lo bf16 pair
 * (2 * y2_conv1_u8_packed_weight_elems() elements from y2_pack_weights_conv1_u8_split).  y bf16 [N,H/2,W/2,64] =
 * [hi(32) | lo(32)] per pixel (the Y2_CONV_IN_SPLIT input layout of the next layer). */
int y2_pack_weights_conv1_u8_split(const float* w_hwio, const float* scale, void* w_packed, y2_stream_t stream);
int y2_conv1_u8_pool_fwd_split(const uint8_t* img, const void* w_packed, const float* shift, void* y, int N, int H, int W,
                               float alpha, y2_stream_t stream);

/* ---- a2: batch normalisation pieces (darknet.py:42-44, tf.layers.batch_normalization) -------
 * y2_bn_stats: per-channel mean and BIASED variance over the M rows of x [M, ld] (float32),
 * accumulated in float64 (activations reach 1e9+ with the reference's initialiser; see DESIGN).
 * workspace: y2_bn_stats_workspace_bytes(M, C) bytes. */
size_t y2_bn_stats_workspace_bytes(int M, int C);
int y2_bn_stats(const float* x, int M, int C, int ld, float* mean, float* var,
                void* workspace, size_t workspace_bytes, y2_stream_t stream);
/* y2_bn_stats plus, in the same finalising kernel, the folded affine of the centred form
 * y = (x - mean) * scale + shift: scale = gamma * rsqrt(var + eps), shift = beta (what y2_bn_fold
 * gives for mean = 0, bias = NULL) -- the training=True branch of darknet.py:42-44 in two launches. */
int y2_bn_stats_fold(const float* x, int M, int C, int ld, float* mean, float* var, const float* gamma,
                     const float* beta, float eps, float* scale, float* shift,
                     void* workspace, size_t workspace_bytes, y2_stream_t stream);
/* ... and the UPDATE_OPS of the training step (pascal_train_darknet.py:49-50) in the same finalising kernel:
 * moving = moving * momentum + batch * (1 - momentum) -- batch statistics of a training layer in two launches. */
int y2_bn_stats_fold_train(const float* x, int M, int C, int ld, float* mean, float* var, const float* gamma, const float* beta,
                           float eps, float* scale, float* shift, float* moving_mean, float* moving_var, float momentum,
                           void* workspace, size_t workspace_bytes, y2_stream_t stream);
/* scale = gamma * rsqrt(var + eps); shift = beta + (bias_or_0 - mean) * scale.
 * Pass conv_bias when the scale/shift is applied to a bias-free accumulator (fused epilogue),
 * NULL when it is applied to h = conv + b. */
int y2_bn_fold(const float* gamma, const float* beta, const float* mean, const float* var,
               const float* conv_bias, float eps, float* scale, float* shift, int C, y2_stream_t stream);
/* moving = moving * momentum + batch * (1 - momentum)   (UPDATE_OPS, pascal_train_darknet.py:49-50) */
int y2_bn_update_moving(float* moving_mean, float* moving_var, const float* mean, const float* var,
                        float momentum, int C, y2_stream_t stream);
/* y = leaky((x - sub) * scale + shift) with optional 2x2 max-pool (darknet.py:45, :24-25); sub,
 * scale, shift are per-channel [C] and may each be NULL (0, 1, 0).  Batch-stat BN passes sub = mean,
 * scale = gamma*rsqrt(var+eps), shift = beta so that the subtraction happens before the scaling.
 * x float32 [N,H,W,C] rows of stride ldx; out_dtype 0: float32, 1: bf16; output [N,Ho,Wo,C] dense. */
int y2_affine_leaky_pool(const float* x, int ldx, const float* sub, const float* scale, const float* shift, float alpha,
                         int leaky, int pool, void* out, int out_dtype, int N, int H, int W, int C,
                         y2_stream_t stream);

/* Same, with an output row stride `ldo` (elements; the result may be a channel slice of a wider, concatenated tensor)
 * and, with space_to_depth != 0, the passthrough / reorg layer (absent from the reference, SURVEY Appendix A) folded
 * into the store address: tf.space_to_depth(block_size=2) semantics, pixel (h, w) -> row (h/2, w/2), channels
 * [((h%2)*2 + (w%2))*C, +C).  `out` then points at the first channel of the slice inside [N, H/2, W/2, ldo].
 * out_dtype 2 = bf16 "hi | lo" pair (the bf16x3 precision mode, see Y2_CONV_IN_SPLIT): hi = bf16(v) at column c and
 * lo = bf16(v - hi) at column lo_off + c of the same row (lo_off 0 -> C, or ldo/2 with space_to_depth); ldo 0 -> 2*C. */
int y2_affine_leaky_pool_ex(const float* x, int ldx, const float* sub, const float* scale, const float* shift, float alpha,
                            int leaky, int pool, void* out, int out_dtype, int ldo, int space_to_depth, int lo_off, int N,
                            int H, int W, int C, y2_stream_t stream);
/* a3: tf.nn.max_pool 2x2/2 (darknet.py:24-25) on bf16 [N,H,W,C] -> [N,H/2,W/2,C]; C % 8 == 0.  (The pool normally runs
 * in the conv epilogue; this kernel serves the layer whose un-pooled output is also the passthrough source.) */
int y2_maxpool2x2_bf16(const void* x, void* y, int N, int H, int W, int C, y2_stream_t stream);
/* tf.nn.avg_pool / tf.layers.average_pooling2d with ksize == stride, evenly divisible map (darknet.py:28-29,116: the
 * 7x7 global pool of the darknet19 classifier).  x NHWC (x_dtype 0 = f32, 1 = bf16) -> y f32 [N,H/k,W/k,C]. */
int y2_avgpool(const void* x, int x_dtype, float* y, int N, int H, int W, int C, int k, y2_stream_t stream);
/* dtype plumbing of the drop-in builders: x_dtype / y_dtype 0 = float32, 1 = bf16 (they must differ); n elements. */
int y2_cast(const void* x, int x_dtype, void* y, int y_dtype, size_t n, y2_stream_t stream);
/* y = x * (*scalar), scalar in DEVICE memory -- the chain rule of get_loss's backward (d loss/d net times the upstream
 * gradient of the scalar loss) without a host synchronisation. */
int y2_scale_by_device_scalar(const float* x, const float* scalar, float* y, size_t n, y2_stream_t stream);

/* ---- a8: grid decode of show_yolo_detection (yolo2_nets/net_utils.py:393-407,418) -----------
 * net [N,S,S,C+5B] f32.  boxes [N,S,S,B,4] = ((x+j)/S, (y+i)/S, w^2, h^2); conf [N,S,S,B];
 * keep [N,S,S,B] u8 = conf > thresh; cls [N,S,S] int32 = argmax of the cell's class vector. */
int y2_decode_ref_v1(const float* net, int N, int S, int B, int C, float thresh,
                     float* boxes, float* conf, uint8_t* keep, int32_t* cls, y2_stream_t stream);

/* ---- a': region decode (YOLOv2; absent from the reference, SURVEY Appendix A) ---------------
 * net [N,S,S,A*(5+C)] f32; anchors [A,2] (cell units).  boxes [N,S*S*A,4] (cx,cy,w,h normalised),
 * scores [N,S*S*A,C] = sigmoid(to)*softmax(c) where > thresh else 0.  One warp per cell. */
int y2_decode_region(const float* net, const float* anchors, int N, int S, int A, int C, float thresh,
                     float* boxes, float* scores, y2_stream_t stream);

/* ---- a': per-class greedy NMS (absent from the reference; IoU arithmetic = net_utils.py:222-260)
 * boxes [N,nbox,4], scores [N,nbox,C].  Candidates of class k: score > score_thresh, visited by
 * (score desc, box index asc); suppressed iff an earlier kept candidate has IoU > iou_thresh.
 * keep_idx [N,C,max_keep] int32 (visiting order; only the first keep_count entries are written),
 * keep_count [N,C] int32 (may exceed max_keep: then only max_keep were stored). */
size_t y2_nms_workspace_bytes(int N, int nbox, int C);
int y2_nms(const float* boxes, const float* scores, int N, int nbox, int C, float score_thresh,
           float iou_thresh, int32_t* keep_idx, int32_t* keep_count, int max_keep,
           void* workspace, size_t workspace_bytes, y2_stream_t stream);

/* ---- a': decode + threshold + per-class NMS fused, one CTA per image (same results as y2_decode_region + y2_nms) -
 * net [N,S,S,A*(5+C)] f32 -> boxes [N,S*S*A,4]; scores [N,S*S*A,C] dense thresholded scores (optional, NULL to skip;
 * needed for the overflow path: images where one class has > 64 candidates are re-done by the y2_nms kernel -- without `scores`
 * such images report keep_count = -1); keep_idx [N,C,max_keep], keep_count [N,C]; keep_score [N,C,max_keep]
 * (optional) = score of each kept box.  C must be 20 and S*S*A <= 4095. */
int y2_detect_fused(const float* net, const float* anchors, int N, int S, int A, int C, float score_thresh,
                    float iou_thresh, float* boxes, float* scores, int32_t* keep_idx, int32_t* keep_count,
                    float* keep_score, int max_keep, y2_stream_t stream);

/* Same contract and results as y2_detect_fused, as two launches sized for the HBM roofline (detect_split.cu): a decode
 * kernel over 32-cell chunks of the whole batch (bulk-copy staged, candidates appended to per-(image, class) lists in the
 * workspace) and a per-image NMS kernel over those lists.  workspace: y2_detect_workspace_bytes(N, C) bytes, 256-byte
 * aligned, ZERO-FILLED once before its first use (every call leaves it zero-filled again).  C == 20, A == 5,
 * S*S*A <= 4095, net / scores 16-byte aligned. */
size_t y2_detect_workspace_bytes(int N, int C);
int y2_detect_split(const float* net, const float* anchors, int N, int S, int A, int C, float score_thresh,
                    float iou_thresh, float* boxes, float* scores, int32_t* keep_idx, int32_t* keep_count,
                    float* keep_score, int max_keep, void* workspace, size_t workspace_bytes, y2_stream_t stream);

/* ---- a7: IoU of n box pairs (yolo2_nets/net_utils.py:222-260 get_iou) ------------------------
 * boxes1/boxes2 [n,4] (cx,cy,w,h) f32 -> iou [n]; float32 in the reference's op order. */
int y2_iou(const float* boxes1, const float* boxes2, float* iou, size_t n, y2_stream_t stream);

/* ---- a6+a7: YOLO loss forward + backward, one kernel (net_utils.py:263-372 + TF autodiff) ----
 * net [N,S,S,C+5B], labels [N,S,S,5+C] float32.  terms[5] = class, coord, object, noobject, total
 * (each already the batch mean, lambda applied).  ious/object_mask [N,S,S,B]; dnet like net
 * (d total / d net).  Any of ious, object_mask, dnet may be NULL.  No pre-zeroing needed: block
 * partials are folded in a fixed order by a trailing 1-block launch (deterministic). */
size_t y2_loss_v1_workspace_bytes(int N, int S);
int y2_loss_v1_fwd_bwd(const float* net, const float* labels, int N, int S, int B, int C,
                       float image_size, float lambda_coord, float lambda_noobj, float* terms,
                       float* ious, float* object_mask, float* dnet,
                       void* workspace, size_t workspace_bytes, y2_stream_t stream);
/* net_utils.py:337-342,366-369: the UNMASKED box deltas the reference logs as histograms ('boxes_delta_x/y/w/h'):
 * predicted (x, y, sqrt w, sqrt h) minus the cell-relative ground truth, every cell and predictor.  deltas [N,S,S,B,4]. */
int y2_loss_v1_box_deltas(const float* net, const float* labels, int N, int S, int B, int C, float image_size, float* deltas,
                          y2_stream_t stream);

/* ---- a': YOLOv2 region loss forward + backward, one kernel (absent from the reference; SURVEY Appendix A) ---
 * net [N,S,S,A*(5+C)] f32; anchors [A,2] (cell units); gt_boxes [N,G,4] normalised (cx,cy,w,h), 16-byte aligned;
 * gt_classes [N,G] int32; gt_counts [N] int32 (<= G).  terms[5] = coord, obj, noobj, class, total (batch means);
 * dnet like net (may be NULL).  Anchor<->ground-truth assignment, IoU, all four terms and the analytic gradient
 * are evaluated per cell by one warp; deterministic reduction. */
size_t y2_region_loss_workspace_bytes(int N, int S);
int y2_region_loss_fwd_bwd(const float* net, const float* anchors, const float* gt_boxes, const int32_t* gt_classes,
                           const int32_t* gt_counts, int N, int S, int A, int C, int G, float lambda_coord,
                           float lambda_obj, float lambda_noobj, float lambda_class, float ignore_thresh, float* terms,
                           float* dnet, void* workspace, size_t workspace_bytes, y2_stream_t stream);

/* ---- a11: backward pass of conv_bn_layer (+ max_pool) -- TF autodiff of darknet.py:39-46, :24-25 ----------
 * y2_bn_leaky_pool_bwd: dy = gradient of the layer output [N,Ho,Wo,C] (dy_dtype 0: float32, 1: bf16; Ho = H/2 when
 * pool).  h_raw = the saved float32 pre-BN rows [N*H*W, ldh] (conv + bias), mean/var = the batch statistics of the
 * forward pass.  Produces dgamma[C], dbeta[C] and dh = d loss / d h_raw as bf16 rows [N*H*W, ld_dh] (columns
 * C..ld_dh-1 zero) -- the operand of both y2_conv_fwd_bf16 (data gradient) and y2_conv_wgrad_bf16.  z, x_hat and the
 * pooling arg-max (first maximum in (dy,dx) scan order) are recomputed from h_raw.  The conv bias gradient is
 * sum(dh) == 0 analytically (a bias in front of a batch-statistics BN is cancelled by the mean subtraction). */
size_t y2_bn_bwd_workspace_bytes(int M, int C);
int y2_bn_leaky_pool_bwd(const float* h_raw, int ldh, const void* dy, int dy_dtype, const float* mean, const float* var,
                         const float* gamma, const float* beta, float eps, float alpha, int leaky, int pool, int N,
                         int H, int W, int C, float* dgamma, float* dbeta, void* dh_bf16, int ld_dh, void* workspace,
                         size_t workspace_bytes, y2_stream_t stream);
/* y2_bn_leaky_pool_bwd_ex: the same, with three ways to read dy (y2_bn_leaky_pool_bwd is this call with ldy = C,
 * dy_s2d = 0, dy_add = NULL, and gives the same bits):
 *   ldy     row stride of dy (>= C; >= 4C with dy_s2d); dy points at the layer's first column, so a channel slice of a
 *           wider gradient (conv2's 1024 columns of the [N,S,S,1280] concat gradient of the YOLOv2 passthrough graph) is
 *           read in place.
 *   dy_s2d  (un-pooled layers, H and W even) the layer's output was stored space_to_depth(2) into rows of stride ldy:
 *           pixel (h, w), channel c is read from row (h/2, w/2), column ((h%2)*2 + w%2)*C + c -- depth_to_space of the
 *           concat gradient, for the passthrough conv.
 *   dy_add  (pooled layers; NULL = none) bf16 [N,H,W,C]: the gradient of the UN-pooled output from a second consumer
 *           (the passthrough branch reads layer 13 before its pool).  Every input row gets its dy_add value, the window's
 *           first maximum also gets the pooled dy; the float32 sum takes that row's leaky slope. */
int y2_bn_leaky_pool_bwd_ex(const float* h_raw, int ldh, const void* dy, int dy_dtype, int ldy, int dy_s2d,
                            const void* dy_add, const float* mean, const float* var, const float* gamma, const float* beta,
                            float eps, float alpha, int leaky, int pool, int N, int H, int W, int C, float* dgamma,
                            float* dbeta, void* dh_bf16, int ld_dh, void* workspace, size_t workspace_bytes,
                            y2_stream_t stream);
/* Data gradient = the forward convolution of dh with the weights transposed (Cin <-> Cout) and flipped spatially:
 * pack them with this, then call y2_conv_fwd_bf16 with Cin := ld_dh, Cout := Cin, no scale/shift/leaky. */
size_t y2_conv_packed_weight_dgrad_elems(int ksize, int Cin, int ld_dh);
int y2_pack_weights_dgrad_bf16(const float* w_hwio, void* w_packed, int ksize, int Cin, int Cout, int ld_dh,
                               y2_stream_t stream);
/* Weight gradient on tcgen05 (both operands MN-major from NHWC via TMA, split-K, fp32 reduction):
 * dw HWIO [k,k,Cin,Cout] float32 += sum_pixels x (bf16 [N,H,W,Cin]) (x) dh (bf16 [N*H*W, ld_dh]).
 * The caller zeroes dw.  Cin % 32 == 0, ld_dh % 64 == 0. */
int y2_conv_wgrad_bf16(const void* x, const void* dh, int ld_dh, float* dw, int N, int H, int W, int Cin, int Cout,
                       int ksize, y2_stream_t stream);
/* First layer (Cin = 3 stored as bf16 [N,H,W,8], 3x3, Cout <= 32): FFMA kernel, dw [3,3,3,Cout] +=. */
int y2_conv_wgrad_c3(const void* x_bf16c8, const void* dh_bf16, int ld_dh, int N, int H, int W, int Cout, float* dw,
                     y2_stream_t stream);
/* out[c] += sum over the M rows of a bf16 matrix [M, ld] (checks sum(dh) ~ 0; bias gradients of BN-free layers). */
int y2_sum_rows_bf16(const void* a_bf16, int ld, size_t M, int C, float* out, y2_stream_t stream);

/* ---- a11: Adam (tf.train.AdamOptimizer defaults, pascal_train_darknet.py:51) -----------------
 * p -= lr_t * m / (sqrt(v) + eps), lr_t = lr * sqrt(1-b2^t)/(1-b1^t) computed by the caller. */
int y2_adam_step(float* p, const float* g, float* m, float* v, size_t n, float lr_t, float beta1,
                 float beta2, float eps, y2_stream_t stream);
/* The training step's form: g is scaled by grad_scale on the fly (1/world of the data-parallel mean), the step size comes
 * from device memory when lr_t_dev != NULL (a CUDA graph of the step then carries no iteration-dependent constant), and
 * with zero_grad != 0 the gradient arena is cleared behind the read (the weight-gradient kernels accumulate into it).
 * n % 4 == 0, all pointers 16-byte aligned. */
int y2_adam_step_ex(float* p, float* g, float* m, float* v, size_t n, float lr_t, const float* lr_t_dev, float beta1,
                    float beta2, float eps, float grad_scale, int zero_grad, y2_stream_t stream);


/* ---- f4: the ImageNet classifier's training graph (src/imagenet/imagenet_train_darknet.py:46-61) ----------------------
 * logits = average over the HW positions of net[N,HW,C] (darknet.py:116-117; HW = 1 for ready-made logits),
 * losses[n] = tf.nn.sparse_softmax_cross_entropy_with_logits (:50-51), correct[n] = (argmax == label) (:60),
 * terms[0] = reduce_mean(losses) (:52), terms[1] = accuracy (:61); dnet (optional, [N,HW,C]) = d terms[0] / d net;
 * logits (optional, [N,C]).  Two launches. */
int y2_softmax_xent_fwd_bwd(const float* net, const int* labels, int N, int HW, int C, float* logits, float* losses,
                            float* correct, float* terms, float* dnet, y2_stream_t stream);
/* tf.train.MomentumOptimizer(lr, momentum) (:58): accum = momentum * accum + g * grad_scale; p -= lr * accum; same
 * conventions as y2_adam_step_ex (n % 4 == 0, 16-byte aligned, zero_grad clears g behind the read). */
int y2_momentum_step(float* p, float* g, float* accum, size_t n, float lr, float momentum, float grad_scale, int zero_grad,
                     y2_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* YOLO2_B200_H_ */
