/* y5obb.h — C ABI of the B200-native yolov5_obb hot path (liby5obb.so).
 *
 * Plain pointers and sizes only; every pointer is a DEVICE pointer unless its name ends in _host.
 * All entry points are asynchronous on `stream` (a cudaStream_t passed as void*) unless stated, never
 * call cudaDeviceSynchronize, and return 0 on success or a Y5OBB_E* code (the Python shims raise
 * RuntimeError on != 0, as the reference's AT_ASSERTM / AT_CUDA_CHECK do).
 *
 * Each declaration cites the reference interface it replaces (paths relative to /root/reference).
 */
#ifndef Y5OBB_H_
#define Y5OBB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Y5OBB_OK 0
#define Y5OBB_EINVAL 1     /* bad argument (null pointer, negative size, unsupported shape) */
#define Y5OBB_EWORKSPACE 2 /* workspace too small: call the matching *_workspace_bytes */
#define Y5OBB_ECUDA 3      /* a CUDA call failed; y5obb_last_cuda_error() has the cudaError_t */
#define Y5OBB_EARCH 4      /* device is not sm_100 */

/* ---- library ------------------------------------------------------------------------------- */
int y5obb_abi_version(void);            /* bumps when a signature, an entry point or a flag is changed or removed */
int y5obb_last_cuda_error(void);        /* cudaError_t of the last failing CUDA call on this thread */
const char* y5obb_build_info(void);     /* "sm_100a nvcc <ver> <date>" */

/* ---- rotated NMS ---------------------------------------------------------------------------
 * Replaces  utils/nms_rotated/src/nms_rotated_ext.cpp:25-39  (nms_rotated(dets, scores, thr))
 *           utils/nms_rotated/src/nms_rotated_cuda.cu:71-134 (sort, 64x64 IoU bit-matrix, D2H, host scan)
 *           utils/nms_rotated/nms_rotated_wrapper.py:26-42   (min(w,h) < 0.001 pre-filter)
 * Everything — sort, IoU tiles, greedy scan, compaction — runs on the device; nothing is copied to
 * the host.
 *
 * flags */
#define Y5OBB_NMS_STRICT_GT 1   /* suppress if IoU >  thr (reference CUDA, nms_rotated_cuda.cu:60); else */
                                /* suppress if IoU >= thr (reference CPU, nms_rotated_cpu.cpp:55)         */
#define Y5OBB_NMS_DROP_SMALL 2  /* boxes with min(w,h) < 0.001 never enter NMS (nms_rotated_wrapper.py:32) */
#define Y5OBB_NMS_NO_CLASS_SPLIT 4  /* y5obb_nms_obb_f32 only: run ONE greedy pass per image over the class-offset boxes
                                       exactly as general.py:849-853 does, instead of independent (image, class)
                                       passes.  The split is the default when classes are offset (not agnostic); it
                                       gives the same rows whenever boxes of different classes cannot overlap, which
                                       the kernel verifies per box (r + max(|cx|,|cy|) < max_wh/2 - 8); if the test
                                       fails counts[batch] comes back as -2 and the caller re-runs with this flag */

#define Y5OBB_NMS_COMPACT_PRED 8     /* y5obb_nms_obb_f32 only: `pred` holds the Detect epilogue's compact records
                                       [batch, anchors, ((nc + 6) + 3) / 4 * 4] = (cx, cy, w, h, obj, cls[nc], theta index, pad)
                                       instead of the [batch, anchors, no] tensor (y5obb_conv_desc.det_decode = 2).  The theta
                                       index is the first maximum of the 180 theta LOGITS (= torch.max over their sigmoids,
                                       utils/general.py:822, whenever those are distinct) */

/* Workspace needed for n_total boxes over n_images images with at most max_per_image boxes in any one
 * image (pass n_total if unknown). */
size_t y5obb_nms_workspace_bytes(int64_t n_total, int64_t n_images, int64_t max_per_image);

/* One NMS problem.  dets5 [n,5] = (cx, cy, w, h, theta_rad) fp32 row-major, scores [n] fp32.
 * keep_out [n] int64 receives indices into dets5 in descending-score order (ties: lower index first);
 * n_keep_out [1] int64 receives the count. */
int y5obb_nms_rotated_f32(const float* dets5, const float* scores, int64_t n, float iou_thr, int flags,
                          int64_t* keep_out, int64_t* n_keep_out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* n_images independent problems in one launch sequence.  image_ids [n_total] int32 in [0, n_images)
 * (any order).  Image b's kept indices (into dets5) are written in descending-score order to
 * keep_out[seg_off_out[b] .. seg_off_out[b] + n_keep_out[b]); seg_off_out has n_images + 1 entries.
 * max_keep > 0 stops each image after that many keeps (non_max_suppression_obb's max_det,
 * utils/general.py:854-855); 0 = unlimited. */
int y5obb_nms_rotated_batched_f32(const float* dets5, const float* scores, const int32_t* image_ids,
                                  int64_t n_total, int64_t n_images, int64_t max_per_image,
                                  float iou_thr, int flags, int64_t max_keep,
                                  int64_t* keep_out, int64_t* n_keep_out, int64_t* seg_off_out,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* Profiling aid for the single-pass NMS (y5obb_nms_rotated[_batched]_f32): with timing on, CUDA events are recorded on the
 * caller's stream between the stages; y5obb_nms_debug_stage_ms then returns {key+radix sort, segments/plan/prep, k_tiles
 * (pairwise IoU bit matrix), k_reduce (greedy scan + compaction)} of the most recent call in milliseconds. */
int y5obb_nms_debug_stage_timing(int on);
int y5obb_nms_debug_stage_ms(float* ms4);

/* Pairwise rotated IoU of n independent pairs (a[i], b[i]), each 5 floats.  Device restatement of
 * utils/nms_rotated/src/box_iou_rotated_utils.h:334-360 (single_box_iou_rotated<float>). */
int y5obb_rbox_iou_pairs_f32(const float* a5, const float* b5, float* iou_out, int64_t n, void* stream);

/* non_max_suppression_obb on the device (utils/general.py:772-862): conf filter, conf = obj*cls, theta =
 * (argmax(180) - 90)/180*3.141592, multi-label expansion, optional class filter (class_mask bit j = class j
 * allowed; ~0 = all), per-image top-max_nms clamp, class offset cls*max_wh on the centre, rotated NMS,
 * max_det.  pred is the Detect eval output [batch, anchors, no] fp32.  Output: out7 [batch, max_det, 7] rows
 * (cx, cy, l, s, theta, conf, cls) in descending-score order, counts [batch + 1] int64 = rows per image, then
 * the total number of candidates found (if > max_candidates the result is incomplete: call again with a
 * larger max_candidates; the Python shim does).  Nothing is synchronised or copied to the host. */
size_t y5obb_nms_obb_workspace_bytes(int64_t batch, int64_t anchors, int64_t max_candidates, int64_t max_nms);
int y5obb_nms_obb_f32(const float* pred, int64_t batch, int64_t anchors, int no, int nc, float conf_thres,
                      float iou_thres, uint64_t class_mask, int agnostic, int multi_label, int max_det, int max_nms,
                      float max_wh, int flags, int64_t max_candidates, float* out7, int64_t* counts,
                      void* workspace, size_t workspace_bytes, void* stream);


/* ---- convolution (tcgen05 implicit GEMM) ---------------------------------------------------
 * Replaces the cuDNN/ATen calls behind models/common.py:37-49 (Conv.forward_fuse = conv + folded-BN
 * bias + SiLU), :94-104 (Bottleneck residual), :267-274 (Concat, as a channel-offset store),
 * nn.Upsample(2x nearest) (models/yolov5*.yaml head) and models/yolo.py:49-81 (Detect).
 * Activations are NHWC bf16; a tensor argument is a channel SLICE of a wider buffer: `ptr` points at
 * the slice's first channel of pixel 0 and `*_pix_stride` is the element distance between pixels.
 * Weights are bf16 packed [KH*KW][cout_pad][cin_pad] (K-major), bias fp32 [cout_pad + 32]
 * (the epilogue reads it in 32-wide chunks); the paddings and
 * the tile shape come from y5obb_conv_tiling so that host packing and kernel agree. */
typedef struct y5obb_conv y5obb_conv_t;

#define Y5OBB_CONV_MODE_CONV 0    /* bf16 NHWC output (+ optional residual / 2x up-sampled copy) */
#define Y5OBB_CONV_MODE_DETECT 1  /* Detect head: fp32 [B, rows, no] output, optional sigmoid+decode */

/* flags: any bit not defined here makes y5obb_conv_create return Y5OBB_EINVAL */
#define Y5OBB_CONV_NO_ROWSHIFT 1   /* flags: force one TMA load per tap (debug / A-B comparison) */
#define Y5OBB_CONV_NO_RESIDENT 2   /* flags: always stream the weight tiles */
#define Y5OBB_CONV_BIAS_HALVED 8    /* flags: REQUIRED when act = 1: `bias` holds 0.5 * b (SiLU is evaluated as h + h*tanh(h), h = x/2) */
#define Y5OBB_CONV_NO_PAIRW 4      /* flags: stride-2 convs use TMA element strides along W instead of the pixel-pair view */
#define Y5OBB_CONV_NO_UP_TMA 2048  /* flags: the 2x up-sampled copy through per-thread stores (default: four TMA stores of the staged tile) */
#define Y5OBB_CONV_NO_RES_RED 16384 /* flags: when `res` IS `out` (in-place Bottleneck add) the default adds the tile into memory with a TMA
                                      reduce-add (bf16 add at L2: the sum is rounded twice); this flag keeps the epilogue's own fp32 add */

typedef struct {
  const void* in;            /* bf16 NHWC slice */
  int64_t in_pix_stride;     /* elements between horizontally adjacent input pixels */
  int64_t in_row_stride;     /* elements between image rows (0 = Win * in_pix_stride) */
  int64_t in_img_stride;     /* elements between images     (0 = Hin * in_row_stride) */
  int B, Hin, Win, Cin;      /* Cin may exceed in_pix_stride: overlapping windows (the stem's merged-kw view) */
  int hbm_cin;               /* channels really read per pixel, for the byte accounting (0 = Cin) */
  const void* w;             /* packed weights */
  const float* bias;
  int Cout, KH, KW, stride, pad_h, pad_w;
  int mode, act;             /* act: 0 = identity, 1 = SiLU */
  int flags;
  void* out;                 /* bf16 NHWC slice (MODE_CONV) */
  int64_t out_pix_stride;
  const void* res;           /* optional residual slice added after the activation (Bottleneck.add) */
  int64_t res_pix_stride;
  void* out2x;               /* optional second destination receiving the 2x nearest up-sampled result */
  int64_t out2x_pix_stride;
  float* det_out;            /* MODE_DETECT: fp32, row = b*det_rows_per_image + det_row_off + (a*H + h)*W + w */
  int64_t det_rows_per_image, det_row_off;
  int det_no;                /* outputs per anchor (nc + 5 + 180) */
  int det_decode;            /* 1: sigmoid + xy/wh decode (eval branch, yolo.py:71-74); 0: raw logits (train) */
  float det_stride;          /* level stride in pixels */
  float det_anchor[6];       /* anchor (w,h) in pixels for the 3 anchors of this level */
  /* optional output geometry (MODE_CONV only; all 0 = derived / dense): the output has out_h x out_w pixels (rows and
     columns of the input read beyond its extent are zero), and out / res pixels (b, h, w) live at
     b * img_stride + h * row_stride + w * pix_stride (elements).  Used by the data gradient of stride-2 convolutions:
     each output-pixel parity class is a 1- or 2-tap stride-1 convolution of dz written to every other pixel. */
  int out_h, out_w;
  int64_t out_row_stride, out_img_stride, res_row_stride, res_img_stride;
} y5obb_conv_desc;

int y5obb_conv_tiling(int cin, int cout, int mode, int det_no, int* block_k, int* block_n, int* cin_pad,
                      int* cout_pad, int* n_tiles_n);
/* Builds TMA descriptors and launch geometry for fixed buffers (host call, no stream work). */
int y5obb_conv_create(const y5obb_conv_desc* desc, y5obb_conv_t** out);
int y5obb_conv_run(const y5obb_conv_t* conv, void* stream);
int y5obb_conv_info(const y5obb_conv_t* conv, double* flops, double* hbm_bytes, int* grid, int* block_n,
                    int* block_k, int* stages);
void y5obb_conv_destroy(y5obb_conv_t* conv);
/* Profiling aid: CTA 0 of every later run writes clock64() stamps of its producer / MMA / epilogue roles for its first 32
 * tiles into dev_buf ([3][32][8] uint64, device memory; NULL switches it off).  Results are unaffected. */
int y5obb_conv_debug_timestamps(y5obb_conv_t* conv, unsigned long long* dev_buf);

/* ---- HBM-bound helpers around the conv stack -------------------------------------------------
 * y5obb_stem_s2d: NCHW fp32 image [B,3,H,W] -> 2x2 space-to-depth NHWC bf16 [B,H/2,W/2,16] (channel
 * (dy*2+dx)*3 + c, 4 zero channels; rows hold pad_cols untouched (zero) pixels on each side), so that the stem Conv(3, c, 6, 2, 2) of models/yolov5*.yaml (layer 0,
 * models/common.py:37-49) becomes a 3x3/s1/p1 conv for the tensor-core kernel.
 * y5obb_sppf_pool: SPPF's three chained MaxPool2d(5,1,2) (models/common.py:181-196) in one pass over
 * channels [0,C) of an NHWC bf16 buffer, results at channel offsets C, 2C, 3C (replaces torch.cat). */
int y5obb_stem_s2d(const float* x_nchw, void* out_nhwc16, int B, int H, int W, int pad_cols, void* stream);
/* same for a uint8 image, with the caller-side `/ 255` (train.py:299, val.py:187-188) folded in */
int y5obb_stem_s2d_u8(const uint8_t* x_nchw, void* out_nhwc16, int B, int H, int W, int pad_cols, void* stream);
int y5obb_sppf_pool(void* buf, int64_t pix_stride, int B, int H, int W, int C, void* stream);
/* y5obb_stem_s2d_u8 for B tiles cropped from a whole scene, replacing the host crop-and-pad of
 * DOTA_devkit/ImgSplit_multi_process.py:122-132 (saveimagepatches, rate 1) and the channel flip of cv2.imread's BGR pixels.
 * scene_hwc [H][W][3] uint8 BGR (any H, W); origins2 [B][2] int32 (left, up) of each tile x tile window; tile b >= n_valid is
 * written as zeros, as are pixels outside the scene.  out_nhwc16 as y5obb_stem_s2d with H = W = tile.  Bit-identical to
 * flipping and zero-padding the crops on the host and calling y5obb_stem_s2d_u8. */
int y5obb_stem_s2d_scene_u8(const uint8_t* scene_hwc, int H, int W, const int32_t* origins2, int B, int n_valid, int tile,
                            void* out_nhwc16, int pad_cols, void* stream);

/* ---- loss ------------------------------------------------------------------------------------
 * Replaces utils/loss.py:122-192 (ComputeLoss.__call__), :194-275 (build_targets) and utils/metrics.py:201-236
 * (bbox_iou, CIoU).  p[i]: Detect training outputs [B, na, H_i, W_i, no] fp32 (models/yolo.py:65);
 * targets [nt, tcols] fp32 rows (img, cls, cx, cy, l, s, theta, csl[180]) in pixels (utils/datasets.py:643-659).
 * Compact targets (SURVEY 8f rank 2: ship 7-8 floats per box over PCIe instead of 187): tcols == 8 -> column 7 is the row's
 * rotation index int(90 - angle) of utils/rboxs_utils.py:21, evaluated by the caller in fp64 like the reference, and the kernel
 * rebuilds the Circular-Smooth-Label row from it (identical loss, the truncation being the only ill-conditioned step);
 * tcols == 7 -> the index is derived in the kernel from theta (column 6): equal to the reference unless fp32 rounding of
 * theta moves angle across an integer (exact multiples of 1 degree can land on either side).
 * loss1[0] = (lbox + lobj + lcls + ltheta) * B, items4 = (lbox, lobj, lcls, ltheta) after the hyp gains
 * (loss.py:185-192).  backward writes dLoss/dp[i] * grad_loss[0] into grad[i] (dense, same shape as p[i]); it
 * must be given the workspace its forward filled.  Duplicate (b,a,gj,gi) cells: the highest source row wins
 * tobj, as sequential CPU index assignment does (loss.py:159). */
typedef struct {
  const float* p[3];
  float* grad[3];            /* backward only */
  int H[3], W[3];
  float stride[3];
  float anchors[18];         /* Detect.anchors: [nl][na][2] in grid units */
  float balance[3];          /* {4.0, 1.0, 0.4} (loss.py:114) */
  int nl, B, na, no, nc;
  const float* targets;
  int nt, tcols;
  float anchor_t, cp, cn;    /* hyp['anchor_t']; smooth_BCE targets (loss.py:107) */
  float hyp_box, hyp_obj, hyp_cls, hyp_theta;  /* already rescaled as train.py:249-252 does */
  float cls_pw, obj_pw, theta_pw;              /* BCEWithLogitsLoss pos_weight (loss.py:99-101) */
  float csl_sigma;                             /* hyp['csl_radius'] for compact targets (tcols 7 / 8); 0 = 2.0 */
} y5obb_loss_desc;

size_t y5obb_loss_workspace_bytes(const y5obb_loss_desc* desc);
int y5obb_loss_forward(const y5obb_loss_desc* desc, float* loss1, float* items4, void* workspace,
                       size_t workspace_bytes, void* stream);
int y5obb_loss_backward(const y5obb_loss_desc* desc, const float* grad_loss, void* workspace,
                        size_t workspace_bytes, void* stream);

/* ---- post-NMS geometry and CSL targets (one thread per box, fp32, separately rounded ops) -------
 * rbox2poly: utils/rboxs_utils.py:106-126 — [n,5] (cx,cy,l,s,theta) -> [n,8] corner coordinates.
 * poly2hbb:  utils/rboxs_utils.py:147-165 — [n,8] -> [n,4] (xc, yc, w, h) of the axis-aligned hull.
 * scale_polys: utils/general.py:636-650 — in place: x -= pad_x, y -= pad_y, all /= gain (un-letterbox).
 * gaussian_label: utils/rboxs_utils.py:9-26 — Circular-Smooth-Label rows [n, num_class] from angles in degrees
 *   (fp64, as numpy evaluates them); peak at bin num_class/2 - trunc(num_class/2 - angle). */
int y5obb_rbox2poly_f32(const float* rboxes5, float* polys8, int64_t n, void* stream);
int y5obb_poly2hbb_f32(const float* polys8, float* hbb4, int64_t n, void* stream);
int y5obb_scale_polys_f32(float* polys8, int64_t n, float pad_x, float pad_y, float gain, void* stream);
/* poly2rbox (utils/rboxs_utils.py:39-81, whose arithmetic is cv2.minAreaRect): [n,8] fp32 corner points ->
 * [n,5] fp64 (cx, cy, long edge, short edge, theta); theta in [-pi/2, pi/2) with pi = 3.141592 (use_pi) or degrees in [0, 180) */
int y5obb_poly2rbox(const float* polys8, double* rbox5, int64_t n, int use_pi, void* stream);
int y5obb_gaussian_label(const double* angle_deg, float* csl_out, int64_t n, int num_class, double sigma,
                         void* stream);

/* ---- training-mode BatchNorm + SiLU (NHWC bf16) ------------------------------------------------
 * Conv.forward = act(bn(conv(x))) in train mode (models/common.py:45-46; BN eps 1e-3, momentum 0.03,
 * utils/torch_utils.py:160-162).  The conv runs raw (act = 0, zero bias) through y5obb_conv_*; then
 *   y5obb_bn_stats      per-channel sum / sum of squares over npix pixels (fp32; deterministic two-stage reduction:
 *                       block partials in `scratch`, added in block order)
 *   y5obb_bn_finalize   scale = gamma / sqrt(var_biased + eps), shift = beta - mean * scale, mean / invstd saved
 *                       for backward, running statistics updated as torch.nn.BatchNorm2d does (unbiased var)
 *   y5obb_bn_silu_apply y = [res +] act(z * scale + shift) into a channel slice, optional 2x nearest copy (W = image
 *                       width in pixels, needed only for the up-sampled copy) */
int64_t y5obb_bn_scratch_floats(int C);  /* scratch (fp32 elements) the two reductions below need for C channels */
int y5obb_bn_stats(const void* z, int64_t z_pix_stride, int64_t npix, int C, float* sum, float* sumsq, float* scratch,
                   int64_t scratch_floats, void* stream);
/* y5obb_bn_stats + y5obb_bn_finalize in two launches (block partials; ordered reduction + finalisation) */
int y5obb_bn_batch_stats(const void* z, int64_t z_pix_stride, int64_t npix, int C, const float* gamma, const float* beta,
                         float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                         float* mean_out, float* invstd_out, float* scratch, int64_t scratch_floats, void* stream);
int y5obb_bn_finalize(const float* sum, const float* sumsq, int64_t npix, int C, const float* gamma, const float* beta,
                      float eps, float momentum, float* running_mean, float* running_var, float* scale, float* shift,
                      float* mean_out, float* invstd_out, void* stream);
int y5obb_bn_silu_apply(const void* z, int64_t z_pix_stride, int64_t npix, int C, int W, const float* scale,
                        const float* shift, int act, const void* res, int64_t res_pix_stride, void* y,
                        int64_t y_pix_stride, void* y2x, int64_t y2x_pix_stride, void* stream);

/* backward of y = [res +] act(bn(z)): dz (bf16 NHWC) from dy; optional pass-through of dy into the residual branch's
 * gradient (gres, overwritten or accumulated); dgamma / dbeta (fp32, overwritten or accumulated).  sum_du / sum_dux are
 * [C] fp32 scratch. */
int y5obb_bn_silu_bwd(const void* z, int64_t z_pix_stride, const void* dy, int64_t dy_pix_stride, int64_t npix, int C,
                      const float* scale, const float* shift, const float* mean, const float* invstd, int act,
                      float* sum_du, float* sum_dux, void* dz, int64_t dz_pix_stride, void* gres,
                      int64_t gres_pix_stride, int gres_accumulate, float* dgamma, float* dbeta, int param_accumulate,
                      float* scratch, int64_t scratch_floats, void* stream);
/* ---- weight gradient (tcgen05 GEMM over the pixel axis) -------------------------------------------
 * dW[tap][co][ci] (fp32, ACCUMULATED with atomics: zero it first) = sum_{b,ho,wo} dz[b,ho,wo,co] * x[b,s*ho+kh-ph,s*wo+kw-pw,ci].
 * Replaces the cuDNN wgrad autograd calls for models/common.py:37-46 under train.py:333.  Operands are the NHWC bf16
 * gradient / activation buffers themselves (channel slices allowed: pix strides in elements, multiples of 8; rows and
 * images dense).  Any map size; zero padding is implicit. */
typedef struct y5obb_wgrad y5obb_wgrad_t;
typedef struct {
  const void* dz;        /* [B][Ho][Wo][dz_pix_stride] bf16, channels [0, Cout) used */
  int64_t dz_pix_stride;
  const void* x;         /* [B][Hi][Wi][x_pix_stride] bf16, channels [0, Cin) used */
  int64_t x_pix_stride;
  int64_t x_row_stride, x_img_stride;  /* elements; 0 = dense (Wi * x_pix_stride, Hi * row).  With explicit strides
                                          x_pix_stride < Cin is allowed: overlapping pixel windows (the stem reads the
                                          3 horizontal taps x 16 space-to-depth channels as one 48-channel pixel) */
  float* dw;             /* fp32; element (tap, co, ci) at dw[tap*dw_tap_stride + co*dw_co_stride + ci*dw_ci_stride] */
  int64_t dw_tap_stride, dw_co_stride, dw_ci_stride;  /* all 0 = dense [KH*KW][Cout][Cin]; (1, Cin*KH*KW, KH*KW) = the
                                                         nn.Conv2d parameter layout [Cout][Cin][KH][KW] */
  int B, Cout, Ho, Wo, Cin, Hi, Wi;
  int KH, KW, stride, pad_h, pad_w;
  int co_group, co_group_pad;  /* Detect: dz channels come in groups of co_group_pad of which the first co_group are
                                  real (padding rows are skipped): dw row = (co / pad) * group + co % pad.  0 = off */
} y5obb_wgrad_desc;
int y5obb_wgrad_create(const y5obb_wgrad_desc* desc, y5obb_wgrad_t** out);
int y5obb_wgrad_run(const y5obb_wgrad_t* w, void* stream);
void y5obb_wgrad_destroy(y5obb_wgrad_t* w);

/* backward helpers of the training graph (NHWC bf16 gradients):
 *   upsample2x_bwd   nn.Upsample(2x nearest) backward: gdst (+)= 2x2 block sums of gsrc
 *   zero_stuff2x     dst[b,2h,2w,:] = src[b,h,w,:] into a pre-zeroed buffer: the dgrad of a stride-2 conv then is a
 *                    stride-1 conv over it with flipped, transposed weights
 *   maxpool5_bwd     one MaxPool2d(5,1,2) backward step of SPPF (models/common.py:190-196) into an fp32 buffer
 *   add_f32_to_bf16  bf16 slice (+)= fp32 dense buffer
 *   detect_grad_pack loss gradient fp32 [B,na,H,W,no] -> bf16 NHWC [B,H,W,na*bn] (the Detect conv's dz) */
int y5obb_upsample2x_bwd(const void* gsrc, int64_t src_pix_stride, void* gdst, int64_t dst_pix_stride, int64_t npix_dst,
                         int C, int W_dst, int accumulate, void* stream);
int y5obb_zero_stuff2x(const void* src, int64_t src_pix_stride, void* dst, int64_t dst_pix_stride, int64_t npix_src, int C,
                       int W_src, void* stream);
int y5obb_maxpool5_bwd(const void* x_in, int64_t in_pix_stride, const float* gout_f32, const void* gout_bf16,
                       int64_t gout_pix_stride, float* gin_f32, int B, int H, int W, int C, void* stream);
int y5obb_add_f32_to_bf16(const float* src, void* dst, int64_t dst_pix_stride, int64_t npix, int C, int accumulate,
                          void* stream);
int y5obb_detect_grad_pack(const float* g, void* out_nhwc, int B, int na, int H, int W, int no, int bn, void* stream);

/* ---- weight re-packing (every optimiser step, train.py:336) ---------------------------------------
 * fp32 nn.Conv2d parameters [Cout][Cin][KH][KW] -> the bf16 operand layouts the conv kernel's TMA descriptors point at,
 * all layers in one launch.  dst is [taps][rows_pad][cols_pad] bf16 (DETECT_BIAS: fp32 [cols_pad]):
 *   FWD           rows = Cout, cols = Cin                         (y5obb_conv_run forward)
 *   DGRAD         rows = Cin,  cols = Cout, taps flipped          (data gradient = conv with transposed weights)
 *   STEM          the 6x6/s2 stem as a 3x1 conv over the 48-channel space-to-depth window (KH=6,KW=6 in; 3 taps out)
 *   DETECT        rows grouped per anchor: group_real real rows padded to group_pad (models/yolo.py:49-65)
 *   DETECT_DGRAD  rows = Cin, cols grouped per anchor
 *   DETECT_BIAS   fp32 bias, grouped per anchor
 *   DGRAD_S2      data gradient of a 3x3 / stride-2 / pad-1 conv for output-pixel parity (ph, pw) = (group_real >> 1,
 *                 group_real & 1): rows = Cin, cols = Cout, (ph ? 2 : 1) x (pw ? 2 : 1) taps; tap t along an axis of parity 1
 *                 is source tap (t == 0 ? 2 : 0), along an axis of parity 0 source tap 1 */
enum { Y5OBB_PACK_FWD = 0, Y5OBB_PACK_DGRAD = 1, Y5OBB_PACK_STEM = 2, Y5OBB_PACK_DETECT = 3, Y5OBB_PACK_DETECT_DGRAD = 4,
       Y5OBB_PACK_DETECT_BIAS = 5, Y5OBB_PACK_DGRAD_S2 = 6 };
typedef struct y5obb_pack_plan y5obb_pack_plan_t;
typedef struct {
  const float* src;
  void* dst;
  int kind, Cout, Cin, KH, KW, rows_pad, cols_pad, group_real, group_pad;
} y5obb_pack_entry;
int y5obb_pack_plan_create(const y5obb_pack_entry* entries, int n, y5obb_pack_plan_t** out);
int y5obb_pack_plan_run(const y5obb_pack_plan_t* plan, void* stream);
void y5obb_pack_plan_destroy(y5obb_pack_plan_t* plan);

/* ---- fused SGD-Nesterov + EMA step -------------------------------------------------------------------------------
 * train.py:148-162,336-342 + utils/torch_utils.py:304-314 over every tensor in one launch.  group 0/1/2 index the per-step
 * learning-rate table (BatchNorm weights / decayed weights / biases); group -1 = EMA only (floating-point buffers);
 * ema may be NULL. */
typedef struct y5obb_sgd_plan y5obb_sgd_plan_t;
typedef struct {
  float* p;          /* parameter (fp32 master weight), updated in place */
  const float* g;    /* gradient */
  float* mom;        /* momentum buffer */
  float* ema;        /* EMA copy of p, or NULL */
  int64_t n;
  float weight_decay;
  int group;
} y5obb_sgd_entry;
int y5obb_sgd_ema_plan_create(const y5obb_sgd_entry* entries, int n, y5obb_sgd_plan_t** out);
int y5obb_sgd_ema_plan_run(const y5obb_sgd_plan_t* plan, const float* lr3, float momentum, float ema_decay, int first_step,
                           void* stream);
void y5obb_sgd_ema_plan_destroy(y5obb_sgd_plan_t* plan);

/* ---- tile-merge polygon NMS of the DOTA devkit (CPU form, double precision) ---------------------------------------
 * DOTA_devkit/ResultMerge_multi_process.py:62-123 py_cpu_nms_poly_fast over DOTA_devkit/polyiou.cpp:106-128 iou_poly, in
 * double precision without FMA contraction (bit-equal to the reference's g++ build by construction; oracle/poly_ref.py).
 * dets9: [n][9] = x1 y1 x2 y2 x3 y3 x4 y4 score (device).  keep_out: indices in descending score order. */
size_t y5obb_poly_nms_workspace_bytes(int64_t n);
int y5obb_poly_nms_f64(const double* dets9, int64_t n, double thresh, int64_t* keep_out, int64_t* n_keep_out, void* workspace,
                       size_t workspace_bytes, void* stream);
int y5obb_poly_iou_pairs_f64(const double* p8, const double* q8, double* iou_out, int64_t n, void* stream);

/* ---- whole-scene merge of tile detections (double precision) ------------------------------------------------------
 * y5obb_tiles_to_scene_f64 replaces DOTA_devkit/ResultMerge_multi_process.py:175-182 (poly2origpoly, rate 1) over the
 * rbox2poly of val.py:226-232 / utils/rboxs_utils.py:106-126: det7 [n_tiles][max_det][7] (cx, cy, l, s, theta, conf, cls;
 * the packed output of y5obb_nms_obb_f32) with counts[t] valid rows, tile origins2 [n_tiles][2] int32 (left, up) and
 * scene_of [n_tiles] int32 (< 0: padding tile, its rows are ignored) -> dets9_out [n][9] (scene-space polygon + score, tile
 * after tile, row after row; capacity n_tiles * max_det) and seg_out [n] = scene * nc + class.  *n_out = n and
 * seg_hist_out [n_scenes * nc] = rows per segment, on the device.
 * y5obb_poly_nms_segmented_f64 replaces ResultMerge_multi_process.py:183-236 (mergesingle: py_cpu_nms_poly_fast, :62-123,
 * once per (scene, class) file entry): y5obb_poly_nms_f64 run independently on every segment seg_id[i] in
 * [0, n_segments).  seg_counts_host [n_segments] (HOST) = rows per segment, which must match seg_id; it sizes the
 * workspace.  keep_out [n]: kept indices into dets9, segment after segment, each in descending score (ties: lower index
 * first); segment s owns keep_out[seg_offsets_out[s] .. seg_offsets_out[s + 1]).  Y5OBB_EINVAL when a segment has more
 * than 1 638 400 rows (its mask row would not fit the 200 KB shared-memory scan). */
size_t y5obb_tiles_to_scene_workspace_bytes(int n_tiles);
int y5obb_tiles_to_scene_f64(const float* det7, const int64_t* counts, int n_tiles, int max_det, const int32_t* origins2,
                             const int32_t* scene_of, int n_scenes, int nc, double* dets9_out, int32_t* seg_out,
                             int64_t* n_out, int64_t* seg_hist_out, void* workspace, size_t workspace_bytes, void* stream);
size_t y5obb_poly_nms_segmented_workspace_bytes(const int64_t* seg_counts_host, int64_t n_segments);
int y5obb_poly_nms_segmented_f64(const double* dets9, const int32_t* seg_id, int64_t n, const int64_t* seg_counts_host,
                                 int64_t n_segments, double thresh, int64_t* keep_out, int64_t* seg_offsets_out,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ---- post-NMS geometry + validation matching (SURVEY 8f rank 3) ------------------------------------------------------
 * One launch per batch for val.py:226-250 + process_batch (val.py:69-92): detections pred7 [batch, max_det, 7] (the packed
 * output of y5obb_nms_obb_f32, counts[b] valid rows) -> native-space polygons polyn8 [batch, max_det, 8] (rbox2poly +
 * scale_polys) and boxes hbbn4 [batch, max_det, 4] (poly2hbb + xywh2xyxy) (either may be NULL), and correct
 * [batch, max_det, niou] (uint8) against labels7 [n_labels, 7] = (image, cls, cx, cy, l, s, theta) in network-input pixels.
 * scale5 [batch, 5] = (gain, pad_x, pad_y, raw_h, raw_w) per image (shapes[si] of val.py:213).  *overflow_flag is set when an
 * image carries more than 1536 labels (the surplus is ignored). */
int y5obb_val_match_f32(const float* pred7, const int64_t* counts, int batch, int max_det, const float* labels7, int n_labels,
                        const float* scale5, const float* iouv, int niou, uint8_t* correct, float* polyn8, float* hbbn4,
                        int* overflow_flag, void* stream);

/* ---- float polygon NMS / rotated-box overlaps (rows A14, B4) ---------------------------------------------------------
 * Device-pointer forms of  utils/nms_rotated/src/nms_rotated_ext.cpp:42-55 nms_poly -> src/poly_nms_cuda.cu:144-261 (K2),
 * DOTA_devkit/poly_nms_gpu/poly_nms_kernel.cu:214-329 (K3) and poly_overlaps_kernel.cu:283-427 (K4); the float polygon IoU
 * restates the reference's expression by expression (union == 0 -> (inter + 1) / (union + 1)).
 * dets9 [n][9] = x1 y1 x2 y2 x3 y3 x4 y4 score.  presorted = 0: polygons are processed by descending score (stable: ties ->
 * lower index), as nms_poly / poly_gpu_nms do before calling the kernel; 1: in the caller's order (the _poly_nms contract).
 * keep_out: indices into dets9 in processing order.  overlaps [n][k] = IoU(boxes5[i], query5[j]), boxes (cx, cy, w, h, angle). */
size_t y5obb_poly_nms_f32_workspace_bytes(int64_t n);
int y5obb_poly_nms_f32(const float* dets9, int64_t n, float iou_thr, int presorted, int64_t* keep_out, int64_t* n_keep_out,
                       void* workspace, size_t workspace_bytes, void* stream);
int y5obb_poly_overlaps_f32(const float* boxes5, const float* query5, int64_t n, int64_t k, float* overlaps, void* stream);
int y5obb_poly_iou_pairs_f32(const float* p8, const float* q8, float* iou_out, int64_t n, void* stream);
/* The devkit's own C ABI (B4): host pointers in and out, synchronous, default stream, CUDA errors printed to stdout - the
 * signatures of DOTA_devkit/poly_nms_gpu/poly_nms.hpp:9-10 and poly_overlaps.hpp:1.  The library also exports them under the
 * reference's C++ names `_poly_nms` / `_overlaps` (include/y5obb_devkit.hpp), which is what the devkit's .pyx files link. */
void y5obb_devkit_poly_nms(int* keep_out_host, int* num_out_host, const float* polys_host, int polys_num, int polys_dim,
                           float nms_overlap_thresh, int device_id);
void y5obb_devkit_overlaps(float* overlaps_host, const float* boxes_host, const float* query_boxes_host, int n, int k,
                           int device_id);

#ifdef __cplusplus
}
#endif
#endif /* Y5OBB_H_ */
