// roi_box.cuh -- the integer box and the resize + shift core shared by the per-ROI disparity hand-off kernels
// (roi_paste.cu: the image-sized paste forms; roi_points.cu: the point-cloud form).
// Core (structures/disparity.py:39-78, DisparityMap.resize / crop): bilinear align_corners=True resize of the [S,S] map to
// (h, wmax) with h = y2-y1, wmax = max(x2-x1, x2p-x1p), value * wmax / S (as (v / S) * wmax in float), crop to x2-x1 columns.
#pragma once
#include "common.cuh"

namespace idisp {

struct RoiBox { int x1, y1, x2, y2, x1p, x2p; };

__device__ __forceinline__ RoiBox roi_box(const float *__restrict__ lb, const float *__restrict__ rb, int r)
{
  RoiBox b;   // expand_box_to_integer (utils/stereo_utils.py:219-229): floor the top-left, ceil the bottom-right; NOT clamped
  b.x1 = (int)floorf(lb[r * 4 + 0]); b.y1 = (int)floorf(lb[r * 4 + 1]); b.x2 = (int)ceilf(lb[r * 4 + 2]); b.y2 = (int)ceilf(lb[r * 4 + 3]);
  b.x1p = (int)floorf(rb[r * 4 + 0]); b.x2p = (int)ceilf(rb[r * 4 + 2]);
  return b;
}

// resized (not yet shifted) disparity of ROI r at image pixel (y, x) inside its box (disparity.py:39-78 as called at disprcnn3d.py:173-175)
__device__ __forceinline__ float roi_disp_at(const float *__restrict__ d, int S, const RoiBox &b, int y, int x)
{
  const int h = b.y2 - b.y1, w = b.x2 - b.x1, wp = b.x2p - b.x1p, wmax = w > wp ? w : wp;
  const float sh = h > 1 ? (float)(S - 1) / (float)(h - 1) : 0.f, sw = wmax > 1 ? (float)(S - 1) / (float)(wmax - 1) : 0.f;
  const float fy = sh * (float)(y - b.y1), fx = sw * (float)(x - b.x1);
  const int y0 = (int)fy, x0 = (int)fx;
  const int y1 = y0 + (y0 < S - 1 ? 1 : 0), x1 = x0 + (x0 < S - 1 ? 1 : 0);
  const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
  const float v = hy * (hx * __ldg(d + y0 * S + x0) + lx * __ldg(d + y0 * S + x1)) + ly * (hx * __ldg(d + y1 * S + x0) + lx * __ldg(d + y1 * S + x1));
  return __fmul_rn(__fdiv_rn(v, (float)S), (float)wmax);
}

}  // namespace idisp
