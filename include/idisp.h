/* idisp.h -- C-ABI of the B200-native iDispNet hot path (libidisp.so).
 *
 * Drop-in boundary for zju3dv/disprcnn's instance-disparity path.  Every entry point is
 * plain C: raw device (or, where stated, host) pointers, explicit sizes, a cudaStream_t
 * passed as void*, int status return (0 = ok; otherwise idisp_last_error() describes the
 * failure for the calling thread).  Outputs are caller-allocated so the host framework
 * (PyTorch in the reference) keeps ownership of all memory; the library holds no global
 * state apart from plan handles.  There is no CPU fallback anywhere behind this header.
 *
 * Reference interfaces replaced (paths relative to the reference root):
 *   idisp_roi_align_forward ... disprcnn/csrc/ROIAlign.h:11-25 (ROIAlign_forward), bound at
 *                               disprcnn/csrc/vision.cpp:9, called from
 *                               disprcnn/layers/roi_align.py:21; CUDA kernel
 *                               disprcnn/csrc/cuda/ROIAlign_cuda.cu:65-122, launcher :257-299.
 *                               The optional per-channel affine fuses
 *                               disprcnn/modeling/detector/disprcnn3d.py:47-49.
 *   idisp_roi_align_backward .. disprcnn/csrc/ROIAlign.h:27-45; training only -> returns
 *                               IDISP_ERR_UNSUPPORTED like the reference's CPU build (:44).
 *   idisp_cost_volume ......... disprcnn/modeling/psmnet/stackhourglass.py:115-128.
 *   idisp_conv3d .............. one convbn_3d / ConvTranspose3d+BN / Conv3d layer:
 *                               disprcnn/modeling/psmnet/submodule.py:19-22,
 *                               stackhourglass.py:11-30,63-88 (test hook, NCDHW in/out).
 *   idisp_softargmin .......... stackhourglass.py:169-172 + submodule.py:51-57.
 *   idisp_plan_* .............. PSMNet's 3-D stack: stackhourglass.py:63-88 (parameters,
 *                               reference state_dict keys) and :115-174 (eval forward).
 */
#ifndef IDISP_H_
#define IDISP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IDISP_VERSION 2  /* 2: + idisp_extractor_*, idisp_roi_*_paste, idisp_stereo_rois, idisp_plan_forward_host_async / host_wait,
                            idisp_roi_points_count / choice / gather (additions only: every version-2 call is unchanged) */

enum {
  IDISP_OK = 0,
  IDISP_ERR_INVALID = 1,     /* bad argument / shape constraint violated            */
  IDISP_ERR_CUDA = 2,        /* a CUDA runtime/driver call or kernel launch failed   */
  IDISP_ERR_UNSUPPORTED = 3, /* not implemented on this path (e.g. ROIAlign backward) */
  IDISP_ERR_STATE = 4        /* plan not finalised / weights missing                 */
};

/* Arithmetic mode of the 3-D conv stack (never silently downgraded). */
enum {
  IDISP_PREC_FP32 = 0,   /* fp32 storage + fp32 FFMA accumulate on the CUDA cores: parity mode (1e-3 abs), any shape     */
  IDISP_PREC_BF16 = 1,   /* bf16 storage + tcgen05 kind::f16 MMA, fp32 accumulate in TMEM (0.1-0.4 px from the reference) */
  IDISP_PREC_FP16 = 2,   /* IEEE-half storage (11-bit significand), same tensor-core kernels (0.02-0.07 px); needs
                            |activation| < 65504 and tensor-core-supported shapes                                         */
  IDISP_PREC_FP16X2 = 3  /* split precision on the tensor cores: every activation and weight is two IEEE-half words
                            (hi + lo, ~22-bit significand), a product is x_hi*w_hi + x_lo*w_hi + x_hi*w_lo accumulated
                            in banked fp32 TMEM accumulators.  Parity mode at tensor-core speed (measured 4e-5..2.6e-4 px
                            from the reference forward); same shape and range limits as IDISP_PREC_FP16.  The default of
                            the Python PSMNet wrapper's benchmark.                                                        */
};

/* conv layer kinds for idisp_conv3d / the plan's layer table */
enum {
  IDISP_CONV_S1 = 0, /* Conv3d k3 s1 p1                               */
  IDISP_CONV_S2 = 1, /* Conv3d k3 s2 p1                               */
  IDISP_DECONV_S2 = 2 /* ConvTranspose3d k3 s2 p1 output_padding 1     */
};

typedef struct idisp_plan idisp_plan_t;
typedef struct idisp_extractor idisp_extractor_t;

int idisp_version(void);
/* Thread-local description of the last failing call ("" if none). Never NULL. */
const char *idisp_last_error(void);

/* Stereo ROI preparation (replaces the Python loop of DispRCNN3D.prepare_psmnet_input_and_target,
 * disprcnn/modeling/detector/disprcnn3d.py:126-146, and expand_box_to_integer, utils/stereo_utils.py:219-229, which pulls
 * every box to the host with .tolist()).  left_boxes / right_boxes [R,4] f32 (x1,y1,x2,y2), image_index [R] int32 -- device
 * pointers.  Writes the aligned crop rectangles rois_left / rois_right [R,5] f32 (batch_idx,x1,y1,x2,y2: same top/bottom,
 * same width) ready for idisp_roi_align_forward, and -- if non-NULL -- x1_x1p_x2_x2p [4][R] int64 (the x1s, x1ps, x2s, x2ps the
 * caller keeps for the disparity -> depth conversion, disprcnn3d.py:150-153).  Integer arithmetic, bit-exact.
 * Clamping uses the size of the image a box belongs to, as the reference does (left_result[i].width / .height, the UNPADDED
 * BoxList size, disprcnn3d.py:136-141): image_wh = device int32 [n_images][2] (width, height) indexed by image_index; when
 * NULL, every box is clamped with the scalar width / height. */
int idisp_stereo_rois(const float *left_boxes, const float *right_boxes, const int *image_index, int R, int width, int height,
                      const int *image_wh, int n_images, float *rois_left, float *rois_right, long long *x1_x1p_x2_x2p,
                      void *stream);

/* Hand-off of the per-ROI disparity maps iDispNet returns (SURVEY.md 8f row 3).  roi_disp [R,S,S] f32; left_boxes / right_boxes
 * [R,4] f32 -- device pointers; boxes are expanded to integers like utils/stereo_utils.py:219-229 and must lie inside the image.
 * Per ROI (disprcnn/structures/disparity.py:39-78 DisparityMap.resize / crop as called at disprcnn3d.py:173-175): bilinear
 * align_corners=True resize of its map to (y2-y1, max(x2-x1, x2p-x1p)), value / S * width, crop to x2-x1 columns, + (x1 - x1p).
 *   idisp_roi_disparity_paste (DispRCNN3D.roi_disp_postprocess, disprcnn3d.py:161-190): clamp at 0, multiply by the ROI's mask
 *     (masks: [R,H,W] uint8 0/1 or NULL), out [N,H,W] = maximum over the image's ROIs (0 where there is none);
 *     roi_start: device int32 [N+1], ROIs roi_start[n] .. roi_start[n+1]-1 belong to image n.
 *   idisp_roi_depth_paste (PointRCNN.process_input, modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:113-136):
 *     out [R,H,W] = fu_baseline[r] / (disp + 1e-6) inside the ROI's box, 0 elsewhere.
 * Agreement with the reference: fp32 rounding of the interpolation (tests: 2e-5 abs / 1e-5 rel). */
int idisp_roi_disparity_paste(const float *roi_disp, int R, int S, const float *left_boxes, const float *right_boxes,
                              const int *roi_start, int N, const unsigned char *masks, int H, int W, float *out, void *stream);
int idisp_roi_depth_paste(const float *roi_disp, int R, int S, const float *left_boxes, const float *right_boxes,
                          const float *fu_baseline, int H, int W, float *out, void *stream);

/* Per-ROI point clouds for PointRCNN (PointRCNN.process_input_eval + back_project(fix_seed=True),
 * modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:189-242 and :37-85): the point-cloud half of SURVEY.md 8f row 3,
 * without any image-sized map.  Three calls: count (device) -> choice per ROI (host) -> gather (device).
 * Inputs shared by count and gather (device pointers): roi_disp [R,S,S] f32 (iDispNet's per-ROI disparity), mask_probs [R,M,M] f32
 * (mask probabilities of the ROI's class), left_boxes / right_boxes [R,4] f32 (x1,y1,x2,y2), image_index [R] int32 (the image
 * each ROI belongs to), image_wh [n_images][2] int32 (width, height), calib [n_images][7] f64 (fu, fv, cu, cv, tx, ty, fu*b: P2
 * entries as Calibration defines them, utils/kitti_utils.py:27-67, and Calib.stereo_fuxbaseline), all used as fp32 scalars;
 * mask_threshold >= 0 and mask_padding >= 1 are the Masker's (modeling/roi_heads/mask_head/inference.py:91-159).
 *   idisp_roi_points_count: count [R] int32 = n, the number of points of each ROI -- the integer box's pixels inside the pasted
 *     mask, or, when the mask covers none of them, all of the box's pixels (point_rcnn.py:42-43).  Negative codes: -1 the integer
 *     box is not inside its image, -2 a depth inside the box is not finite, -3 image_index out of range.
 *   idisp_roi_points_choice (HOST, no GPU): out [npoints] int32 = the indices numpy draws for n valid points (point_rcnn.py:53-74
 *     with np.random.seed(0) before each draw), bit for bit: choice(n, P, replace=False) if n > P, else arange(n) followed by
 *     choice(n, P - n, replace=True); then shuffled.  n >= 1.
 *   idisp_roi_points_gather: ranks [R,npoints] int32 (device; row r = choice for count[r]) -> pts [R,npoints,3] f32 (rotated about
 *     y by rot_angle, z clamped at max_depth before the rotation, centred), pts_mean [R,3] f32 (the mean that was subtracted),
 *     rot_angle [R] f64 (atan2((x1 + x2) / 2 - W0 / 2, fu), W0 = the width of image 0 as in utils/utils_3d.py:88), and -- if
 *     non-NULL -- pixels [R,npoints] int32 (y * width + x of each point).  A slot whose rank is outside [0, count[r]) (every slot
 *     of a ROI with count[r] <= 0) gets NaN coordinates and pixel -1.  npoints <= 16384.
 * R == 0 is a no-op. */
int idisp_roi_points_count(const float *roi_disp, int R, int S, const float *mask_probs, int M, const float *left_boxes,
                           const float *right_boxes, const int *image_index, const int *image_wh, const double *calib,
                           int n_images, float mask_threshold, int mask_padding, int *count, void *stream);
int idisp_roi_points_choice(int n, int npoints, int *out);
int idisp_roi_points_gather(const float *roi_disp, int R, int S, const float *mask_probs, int M, const float *left_boxes,
                            const float *right_boxes, const int *image_index, const int *image_wh, const double *calib,
                            int n_images, float mask_threshold, int mask_padding, const int *count, const int *ranks,
                            int npoints, float max_depth, float *pts, float *pts_mean, double *rot_angle, int *pixels,
                            void *stream);

/* ROIAlign forward.  input [N,C,H,W] f32 NCHW contiguous, rois [R,5] f32
 * (batch_idx,x1,y1,x2,y2), out [R,C,pooled_h,pooled_w] f32 -- all device pointers.
 * mean/inv_std: optional device pointers to C floats; when non-NULL the kernel writes
 * (v - mean[c]) / std[c] with std[c] passed as-is in `std` (division, like the
 * reference's in-place sub_/div_).  R == 0 is a no-op (reference early-return :278-281). */
int idisp_roi_align_forward(const float *input, int N, int C, int H, int W, const float *rois, int R,
                            float spatial_scale, int pooled_h, int pooled_w, int sampling_ratio,
                            const float *mean, const float *std, float *out, void *stream);
int idisp_roi_align_backward(const float *grad, const float *rois, int R, float spatial_scale,
                             int pooled_h, int pooled_w, int N, int C, int H, int W,
                             int sampling_ratio, float *grad_input, void *stream);

/* Concatenation cost volume.  left/right [B,C,Hf,Wf] f32 NCHW -> cost [B,2C,D,Hf,Wf] f32
 * NCDHW with D=(maxdisp-mindisp)/4; mindisp, maxdisp multiples of 4, |shift| < Wf. */
int idisp_cost_volume(const float *left, const float *right, int B, int C, int Hf, int Wf,
                      int mindisp, int maxdisp, float *cost, void *stream);

/* One 3x3x3 conv layer with folded affine epilogue (per-layer test hook; NCDHW f32 I/O,
 * converted to the internal channel-blocked layout inside).
 *   kind: IDISP_CONV_*.  weight: Conv3d layout [Cout,Cin,3,3,3] (S1,S2) or ConvTranspose3d
 *   layout [Cin,Cout,3,3,3] (DECONV_S2), device f32.  scale/bias: per-Cout f32 device
 *   pointers, y = conv(x)*scale + bias (NULL -> 1 / 0); residual (NULL or NCDHW f32 of the
 *   output shape) is added before the optional ReLU.  precision: IDISP_PREC_*.
 *   Output dims: S1 same; S2 ceil(n/2); DECONV 2n. */
int idisp_conv3d(const float *x, int B, int Cin, int D, int H, int W, const float *weight, int Cout,
                 int kind, const float *scale, const float *bias, const float *residual, int relu,
                 int precision, float *y, void *stream);

/* Trilinear(align_corners) upsample of logits [B,D,Hf,Wf] f32 to [B,maxdisp-mindisp,H,W],
 * softmax over disparity, expectation over d in [mindisp,maxdisp) -> out [B,H,W] f32;
 * the upsampled volume is never materialised. */
int idisp_softargmin(const float *logits, int B, int D, int Hf, int Wf, int mindisp, int maxdisp,
                     int H, int W, float *out, void *stream);

/* ---- plan: the 28-layer stack with reference-keyed weights ------------------------- */
/* C = feature channels per view (dres0.0 has 2C inputs). */
int idisp_plan_create(int C, int mindisp, int maxdisp, int precision, idisp_plan_t **plan);
void idisp_plan_destroy(idisp_plan_t *plan);
/* Hand over one reference state_dict entry by its key (e.g. "dres0.0.0.weight",
 * "dres2.conv5.1.running_var"); data is a HOST pointer to numel f32 values in the reference's
 * own layout.  Unknown keys (feature_extraction.*, *.num_batches_tracked) return IDISP_OK
 * and are ignored, so a whole reference checkpoint can be streamed through. */
int idisp_plan_set_tensor(idisp_plan_t *plan, const char *key, const float *data, size_t numel);
/* Fold BN (eps 1e-5) into per-channel scale/bias, re-lay the kernels for the selected
 * precision, upload.  Fails with IDISP_ERR_STATE naming the first missing key. */
int idisp_plan_finalize(idisp_plan_t *plan, void *stream);
/* Bytes of device workspace idisp_plan_forward needs for this shape. */
size_t idisp_plan_workspace_bytes(const idisp_plan_t *plan, int B, int Hf, int Wf);
/* left/right [B,C,Hf,Wf] f32 NCHW device -> out [B,H,W] f32 device.
 * D, Hf, Wf must be multiples of 4 (two stride-2 stages, stackhourglass.py:34-49). */
int idisp_plan_forward(idisp_plan_t *plan, const float *left, const float *right, int B, int Hf,
                       int Wf, int H, int W, void *workspace, size_t workspace_bytes, float *out,
                       void *stream);
/* fp16-word modes (IDISP_PREC_FP16, IDISP_PREC_FP16X2): did the most recent idisp_plan_forward on this plan produce an
 * activation (or take an input feature) outside the IEEE-half range, |v| > 65504 or non-finite?  Such a value is stored as
 * inf and -- because ReLU's max(NaN, 0) is 0 -- can end in finite but wrong disparities.  Writes 0/1 to *exceeded (host
 * pointer); synchronises `stream`.  Always 0 for fp32 / bf16 plans.  The Python wrapper's precision='auto' uses it to redo such
 * a batch with the fp32 kernels. */
int idisp_plan_range_exceeded(idisp_plan_t *plan, int *exceeded, void *stream);

/* Same call with HOST buffers (pinned recommended): H2D of left/right, forward, D2H of out,
 * all enqueued on `stream`; the plan owns and grows the device staging + workspace. */
int idisp_plan_forward_host(idisp_plan_t *plan, const float *left_host, const float *right_host,
                            int B, int Hf, int Wf, int H, int W, float *out_host, void *stream);
/* Pipelined form for a stream of batches (the reference's loader feeds DispRCNN3D batch after batch, engine/inference.py:24-50):
 * the host->device copy of this call's inputs runs on a plan-owned copy stream and overlaps the kernels of the previous call
 * still running on `stream`; the device->host copy of the result runs on a second copy stream and overlaps the next call's
 * kernels.  Device staging is double-buffered (slot = call parity); the kernels of successive calls stay ordered on `stream`.
 * Never blocks the host.  *ticket identifies the call: out_host (and left_host / right_host for reuse) belong to the library
 * until idisp_plan_host_wait(plan, ticket) has returned. */
int idisp_plan_forward_host_async(idisp_plan_t *plan, const float *left_host, const float *right_host, int B, int Hf,
                                  int Wf, int H, int W, float *out_host, void *stream, unsigned long long *ticket);
/* Blocks the calling host thread until the result of the call that returned `ticket` is in its out_host buffer. */
int idisp_plan_host_wait(idisp_plan_t *plan, unsigned long long ticket);
/* Debug/test hook: copy the low-resolution logits cost3 [B,D,Hf,Wf] f32 of the last
 * idisp_plan_forward on this plan into a device buffer. */
int idisp_plan_get_logits(idisp_plan_t *plan, float *logits, void *stream);
/* Number of kernel launches one idisp_plan_forward enqueues (for bench bookkeeping). */
int idisp_plan_launches_per_forward(const idisp_plan_t *plan);
/* The tensor-core modes capture the conv section of a forward (every launch between the input conversion and the soft-argmin:
 * it touches only the workspace) into a CUDA graph the first time a (B, Hf, Wf, workspace) combination is seen and replay it
 * with one cudaGraphLaunch afterwards (disabled by IDISP_NO_GRAPH=1, while per-launch timing is on, and inside a caller's own
 * stream capture).  Writes how many graphs this plan has captured / how many forwards replayed one (either may be NULL). */
int idisp_plan_graph_stats(const idisp_plan_t *plan, int *captures, int *replays);
/* Per-launch device timing of idisp_plan_forward (CUDA events on the forward's stream between
 * consecutive launches).  After a forward with timing enabled, get_timing writes, for each of the
 * launches_per_forward launches, its duration in ms and the layer it ran (0..27 = SURVEY.md
 * Appendix A order minus one; -1 = cost volume, -2 = soft-argmin).  capacity = array lengths. */
int idisp_plan_enable_timing(idisp_plan_t *plan, int on);
int idisp_plan_get_timing(idisp_plan_t *plan, float *ms, int *layer, int capacity);

/* ---- the 2-D feature extractor that precedes the cost volume in the live call (SURVEY.md 8f row 1) -------------------
 * disprcnn/modeling/psmnet/submodule.py:60-139 (feature_extraction: firstconv, layer1-4 of BasicBlocks :25-48, four SPP
 * branches, concat, lastconv), applied to each view at stackhourglass.py:112-113.  Same pattern as the plan: hand over the
 * reference's state_dict entries by key (relative to the module: "firstconv.0.0.weight", "layer2.0.downsample.1.running_var",
 * "lastconv.2.weight", ...; *.num_batches_tracked is ignored), finalize (BatchNorm2d folded in float64), forward.
 * images [B,3,H,W] f32 NCHW device -> features [B,32,H/4,W/4] f32 NCHW device (H/4 = ((H-1)/2+1-1)/2+1: two k3 s2 p1 convs);
 * H/4 and W/4 must be at least 56 (branch1's 56x56 average pool, submodule.py:78).  fp32 FFMA kernels, no CPU path. */
int idisp_extractor_create(idisp_extractor_t **extractor);
void idisp_extractor_destroy(idisp_extractor_t *extractor);
int idisp_extractor_set_tensor(idisp_extractor_t *extractor, const char *key, const float *data, size_t numel);
int idisp_extractor_finalize(idisp_extractor_t *extractor, void *stream);
size_t idisp_extractor_workspace_bytes(const idisp_extractor_t *extractor, int B, int H, int W);
int idisp_extractor_forward(idisp_extractor_t *extractor, const float *images, int B, int H, int W, void *workspace,
                            size_t workspace_bytes, float *features, void *stream);
int idisp_extractor_launches_per_forward(const idisp_extractor_t *extractor);
/* Arithmetic of the 53 stride-1 3x3 convolutions (99 % of the extractor's FLOPs): IDISP_PREC_FP16X2 (default) = tcgen05 tensor
 * cores in split precision (two IEEE-half words per value, three MMAs per product, fp32 accumulate: fp32-grade, csrc/conv2d_tc.cu);
 * IDISP_PREC_FP32 = the fp32 FFMA kernels for every layer.  Call before idisp_extractor_finalize (a change un-finalises). */
int idisp_extractor_set_precision(idisp_extractor_t *extractor, int precision);
/* IDISP_PREC_FP16X2 only: did the most recent forward see a value outside the IEEE-half range (see idisp_plan_range_exceeded)?
 * Writes 0/1 to *exceeded (host pointer); synchronises `stream`. */
int idisp_extractor_range_exceeded(idisp_extractor_t *extractor, int *exceeded, void *stream);

/* Test hook: the cost volume exactly as the tensor-core path assembles it inside dres0.0's TMA loader (never
 * materialised in the product path): bf16-rounded values, NCDHW f32 out [B,2C,D,Hf,Wf].  C in {16, 32}. */
int idisp_debug_fused_cost_volume(const float *left, const float *right, int B, int C, int Hf, int Wf,
                                  int mindisp, int maxdisp, float *cost, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* IDISP_H_ */
