// roi_paste.cu -- what happens to a per-ROI disparity map right after iDispNet: the hand-off to the full image and to depth
// (SURVEY.md section 8(f) row 3).  Two reference call sites share one core:
//   * DispRCNN3D.roi_disp_postprocess, disprcnn/modeling/detector/disprcnn3d.py:161-190 -- every ROI's [S,S] disparity is
//     resized to its (integer-expanded) box, shifted by x1 - x1p, clamped at 0, masked, pasted into a zero image-sized map, and
//     the per-image map is the maximum over the image's ROIs;
//   * PointRCNN.process_input, modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:113-136 -- the same resize + shift, then
//     depth = fu*baseline / (disp + 1e-6) pasted into a per-ROI image-sized map (which back_project masks and back-projects).
// Core: roi_box / roi_disp_at (roi_box.cuh, shared with roi_points.cu).
// The reference does this per ROI in Python (.tolist() syncs, one image-sized zeros + interpolate + slice-assign per ROI); here
// one thread per image pixel walks the ROIs of its image and samples the low-resolution map directly -- nothing image-sized per
// ROI is materialised in the disparity form.  Integer box arithmetic is exact; the interpolation follows ATen's index math
// (scale = (in-1)/(out-1), i0 = (int)src, lambda = src - i0) so results agree with the reference to fp32 rounding.
// Roofline: HBM (writes N*H*W*4 B, reads the touched parts of the R low-resolution maps from L2).
#include "roi_box.cuh"

namespace idisp {

// per-image disparity map: out[n][y][x] = max over the image's ROIs of clamp(disp, 0) * mask   (disprcnn3d.py:176-183)
// roi_start[n] .. roi_start[n+1]: the ROIs of image n (ROIs are grouped by image, as torch.split(output, ...) assumes, :162)
__global__ void roi_disparity_paste_kernel(const float *__restrict__ disp, int S, const float *__restrict__ lb, const float *__restrict__ rb,
                                           const int *__restrict__ roi_start, const unsigned char *__restrict__ masks, int H, int W,
                                           float *__restrict__ out)
{
  const int n = blockIdx.z, y = blockIdx.y;
  const int r0 = roi_start[n], r1 = roi_start[n + 1];
  for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < W; x += gridDim.x * blockDim.x) {
    float best = 0.f;
    for (int r = r0; r < r1; ++r) {
      const RoiBox b = roi_box(lb, rb, r);
      if (y < b.y1 || y >= b.y2 || x < b.x1 || x >= b.x2) continue;
      if (masks && !masks[((long long)r * H + y) * W + x]) continue;
      const float v = fmaxf(__fadd_rn(roi_disp_at(disp + (long long)r * S * S, S, b, y, x), (float)(b.x1 - b.x1p)), 0.f);   // :178 + clamp :179
      best = fmaxf(best, v);
    }
    out[((long long)n * H + y) * W + x] = best;
  }
}

// per-ROI depth map (point_rcnn.py:124-134): depth[r][y][x] = fub[r] / (disp + 1e-6) inside the box, 0 elsewhere
__global__ void roi_depth_paste_kernel(const float *__restrict__ disp, int S, const float *__restrict__ lb, const float *__restrict__ rb,
                                       const float *__restrict__ fub, int H, int W, float *__restrict__ out)
{
  const int r = blockIdx.z, y = blockIdx.y;
  const RoiBox b = roi_box(lb, rb, r);
  const float f = fub[r];
  for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < W; x += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (y >= b.y1 && y < b.y2 && x >= b.x1 && x < b.x2) {
      // point_rcnn.py:130-131: disp_roi + x1 - x1p (two float adds), fu*baseline / (disp + 1e-6)
      const float d = __fadd_rn(__fadd_rn(roi_disp_at(disp + (long long)r * S * S, S, b, y, x), (float)b.x1), -(float)b.x1p);
      v = __fdiv_rn(f, __fadd_rn(d, 1e-6f));
    }
    out[((long long)r * H + y) * W + x] = v;
  }
}

}  // namespace idisp

using namespace idisp;

static int roi_paste_check(const char *who, int R, int S, int N, int H, int W)
{
  IDISP_REQUIRE(R >= 0 && S > 0 && N >= 0 && H > 0 && W > 0, "%s: bad shape R=%d S=%d N=%d H=%d W=%d", who, R, S, N, H, W);
  IDISP_REQUIRE(H <= 65535 && N <= 65535 && R <= 65535, "%s: H, N and R must fit a CUDA grid dimension (65535)", who);
  return IDISP_OK;
}

extern "C" int idisp_roi_disparity_paste(const float *roi_disp, int R, int S, const float *left_boxes, const float *right_boxes,
                                         const int *roi_start, int N, const unsigned char *masks, int H, int W, float *out, void *stream)
{
  int rc = roi_paste_check("roi_disparity_paste", R, S, N, H, W);
  if (rc) return rc;
  if (N == 0) return IDISP_OK;
  IDISP_REQUIRE(out && roi_start && (R == 0 || (roi_disp && left_boxes && right_boxes)), "roi_disparity_paste: NULL pointer");
  const int threads = 128;
  roi_disparity_paste_kernel<<<dim3(ceil_div(W, threads), H, N), threads, 0, (cudaStream_t)stream>>>(roi_disp, S, left_boxes, right_boxes, roi_start,
                                                                                                     masks, H, W, out);
  IDISP_LAUNCH_CHECK();
  return IDISP_OK;
}

extern "C" int idisp_roi_depth_paste(const float *roi_disp, int R, int S, const float *left_boxes, const float *right_boxes,
                                     const float *fu_baseline, int H, int W, float *out, void *stream)
{
  int rc = roi_paste_check("roi_depth_paste", R, S, 1, H, W);
  if (rc) return rc;
  if (R == 0) return IDISP_OK;
  IDISP_REQUIRE(roi_disp && left_boxes && right_boxes && fu_baseline && out, "roi_depth_paste: NULL pointer");
  const int threads = 128;
  roi_depth_paste_kernel<<<dim3(ceil_div(W, threads), H, R), threads, 0, (cudaStream_t)stream>>>(roi_disp, S, left_boxes, right_boxes, fu_baseline, H, W, out);
  IDISP_LAUNCH_CHECK();
  return IDISP_OK;
}
