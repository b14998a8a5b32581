// roi_points.cu -- per-ROI point clouds for PointRCNN straight from iDispNet's per-ROI disparity maps (SURVEY.md section 8(f) row 3,
// the point-cloud half).  Eval path of PointRCNN.process_input_eval (modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:
// 189-242) and back_project(..., fix_seed=True) (:37-85).  Per ROI, in the reference's order:
//   1. integer boxes (expand_box_to_integer, roi_box.cuh);
//   2. the Masker's mask (modeling/roi_heads/mask_head/inference.py:91-159): [M,M] probabilities padded to M+2p, the float left box
//      scaled by (M+2p)/M about its centre and truncated to int32, bilinear align_corners=False resize to that box, > threshold;
//   3. depth = fu*b / (disp + x1 - x1p + 1e-6) clamped at 1 inside the integer box (:214-219), 0 elsewhere;
//   4. the mask is applied only if it covers some pixel of the integer box (:42-43), otherwise the whole box is kept;
//   5. points through depthmap_to_rect (structures/calib.py:103-122), pixels enumerated column-major (x outer, y inner);
//   6. the valid points (z > 0) sampled to P by numpy's seeded choice + shuffle (:53-74) -- on the host, idisp_roi_points_choice;
//   7. z clamped at max_depth (:84);  8. rotation about y by atan2(cx - W0/2, fu) (utils/utils_3d.py:74-104);  9. centring.
// Two launches around the host sampler: roi_points_count_kernel (steps 1-4: the number n of valid points of every ROI) and
// roi_points_gather_kernel (the chosen ranks -> pixels, steps 5, 7-9).  Nothing image-sized is allocated or written: the reference
// materialises two image-sized maps per ROI and back-projects every pixel of the image.
// Roofline: neither kernel moves more than a few hundred KB; both are latency-bound (one CTA per ROI).
#include <algorithm>
#include <numeric>
#include <vector>

#include "roi_box.cuh"

namespace idisp {

constexpr int PTS_THREADS = 512;
constexpr int PTS_MAX_POINTS = 16384;   // ranks + chosen pixels of one ROI live in shared memory (128 KB)
constexpr int PTS_MAX_MASK = 128;       // padded mask side M + 2 * padding

// calib [N][7] f64, per image
enum { CAL_FU, CAL_FV, CAL_CU, CAL_CV, CAL_TX, CAL_TY, CAL_FUB, CAL_N };

// everything about ROI r that does not depend on the pixel
struct RoiPts {
  RoiBox b;
  int h, w;                  // integer box size (rows, columns)
  int mx0, my0, mx1, my1;    // the Masker's integer box, inclusive corners (inference.py:120-121)
  int mw, mh;                // size of the resized mask (:124-127)
  float msx, msy;            // bilinear scales (M+2p) / mw, (M+2p) / mh
  int Mp;                    // padded mask side
  float thr, fub;
  int img, W, H;
  int status;                // 0, or the negative count code
};

__device__ __forceinline__ RoiPts roi_pts_setup(const float *__restrict__ lb, const float *__restrict__ rb, int r, const int *__restrict__ image_index,
                                                const int *__restrict__ image_wh, const double *__restrict__ calib, int n_images, int M, int pad,
                                                float thr)
{
  RoiPts g;
  g.b = roi_box(lb, rb, r);
  g.h = g.b.y2 - g.b.y1; g.w = g.b.x2 - g.b.x1;
  g.img = image_index[r];
  g.status = 0;
  if (g.img < 0 || g.img >= n_images) { g.status = -3; g.img = 0; }
  g.W = image_wh[2 * g.img]; g.H = image_wh[2 * g.img + 1];
  // the box must be a (possibly empty) rectangle inside the image: the reference slice-assigns depth_map[y1:y2, x1:x2] (:218)
  if (!g.status && (g.b.x1 < 0 || g.b.y1 < 0 || g.b.x2 > g.W || g.b.y2 > g.H || g.w < 0 || g.h < 0)) g.status = -1;
  g.fub = (float)calib[g.img * CAL_N + CAL_FUB];
  g.thr = thr;
  // Masker box (expand_boxes, inference.py:91-106, in float32; the scale is a Python float applied to a float32 tensor)
  g.Mp = M + 2 * pad;
  const float scale = (float)((double)g.Mp / (double)M);
  const float bx0 = lb[r * 4 + 0], by0 = lb[r * 4 + 1], bx1 = lb[r * 4 + 2], by1 = lb[r * 4 + 3];
  const float w_half = __fmul_rn(__fmul_rn(__fsub_rn(bx1, bx0), 0.5f), scale), h_half = __fmul_rn(__fmul_rn(__fsub_rn(by1, by0), 0.5f), scale);
  const float x_c = __fmul_rn(__fadd_rn(bx1, bx0), 0.5f), y_c = __fmul_rn(__fadd_rn(by1, by0), 0.5f);
  g.mx0 = __float2int_rz(__fsub_rn(x_c, w_half)); g.mx1 = __float2int_rz(__fadd_rn(x_c, w_half));   // .to(torch.int32)
  g.my0 = __float2int_rz(__fsub_rn(y_c, h_half)); g.my1 = __float2int_rz(__fadd_rn(y_c, h_half));
  g.mw = max(g.mx1 - g.mx0 + 1, 1); g.mh = max(g.my1 - g.my0 + 1, 1);
  g.msx = __fdiv_rn((float)g.Mp, (float)g.mw); g.msy = __fdiv_rn((float)g.Mp, (float)g.mh);   // area_pixel_compute_scale
  return g;
}

// ATen's align_corners=False source index: scale * (dst + 0.5) - 0.5 clamped at 0, i1 = i0 + (i0 < in - 1)
__device__ __forceinline__ void lin_index(float scale, int dst, int in, int &i0, int &i1, float &l1)
{
  float src = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
  src = src < 0.f ? 0.f : src;
  i0 = min((int)src, in - 1);
  l1 = fminf(fmaxf(__fsub_rn(src, (float)i0), 0.f), 1.f);
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
}

// Pixel (y, x) of ROI r, inside its integer box.  Writes the depth the reference's map holds there (z: clamped at 1, NaN kept) and
// returns whether the Masker's pasted mask covers it.  The ONE definition of a ROI's points both kernels use: the count kernel counts
// with it, the gather kernel ranks with it, so the sampled ranks always index the gather's list.
__device__ __forceinline__ bool roi_pixel(const RoiPts &g, const float *__restrict__ disp, int S, const float *mask_s, int y, int x, float &z)
{
  // point_rcnn.py:214-218: (disp + x1) - x1p, fu*b / (d + 1e-6) as reciprocal * float (Tensor.__rdiv__), clamp(min=1.0)
  const float d = __fadd_rn(__fadd_rn(roi_disp_at(disp, S, g.b, y, x), (float)g.b.x1), -(float)g.b.x1p);
  const float depth = __fmul_rn(__frcp_rn(__fadd_rn(d, 1e-6f)), g.fub);
  z = depth != depth ? depth : fmaxf(depth, 1.f);
  if (y < g.my0 || y > g.my1 || x < g.mx0 || x > g.mx1) return false;
  int y0, y1, x0, x1;
  float ly, lx;
  lin_index(g.msy, y - g.my0, g.Mp, y0, y1, ly);
  lin_index(g.msx, x - g.mx0, g.Mp, x0, x1, lx);
  const float hy = __fsub_rn(1.f, ly), hx = __fsub_rn(1.f, lx);
  const float *m = mask_s;
  const float top = __fadd_rn(__fmul_rn(m[y0 * g.Mp + x0], hx), __fmul_rn(m[y0 * g.Mp + x1], lx));
  const float bot = __fadd_rn(__fmul_rn(m[y1 * g.Mp + x0], hx), __fmul_rn(m[y1 * g.Mp + x1], lx));
  return __fadd_rn(__fmul_rn(top, hy), __fmul_rn(bot, ly)) > g.thr;
}

// expand_masks (inference.py:109-118): the [M,M] probabilities inside a zero border of `pad`
__device__ __forceinline__ void stage_mask(float *mask_s, const float *__restrict__ probs, int M, int pad, int Mp)
{
  for (int i = threadIdx.x; i < Mp * Mp; i += blockDim.x) {
    const int yy = i / Mp - pad, xx = i % Mp - pad;
    mask_s[i] = (yy >= 0 && yy < M && xx >= 0 && xx < M) ? __ldg(probs + yy * M + xx) : 0.f;
  }
}

template <typename T>
__device__ __forceinline__ T block_sum(T v, T *red)
{
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[warp] = v;
  __syncthreads();
  T t = 0;
  for (int i = 0; i < nw; ++i) t += red[i];   // fixed order: the same result on every thread and every call
  return t;
}

// count[r] = n: the number of box pixels inside the mask if there are any, else the number of box pixels (the unmasked fallback);
// -1: integer box not inside its image, -2: a non-finite depth inside the box, -3: image index out of range
__global__ void __launch_bounds__(PTS_THREADS) roi_points_count_kernel(
    const float *__restrict__ disp, int S, const float *__restrict__ probs, int M, int pad, float thr, const float *__restrict__ lb,
    const float *__restrict__ rb, const int *__restrict__ image_index, const int *__restrict__ image_wh, const double *__restrict__ calib,
    int n_images, int *__restrict__ count)
{
  extern __shared__ float mask_s[];
  __shared__ int red[PTS_THREADS / 32];
  const int r = blockIdx.x;
  const RoiPts g = roi_pts_setup(lb, rb, r, image_index, image_wh, calib, n_images, M, pad, thr);
  if (g.status) {
    if (threadIdx.x == 0) count[r] = g.status;
    return;
  }
  stage_mask(mask_s, probs + (long long)r * M * M, M, pad, g.Mp);
  __syncthreads();
  const float *d = disp + (long long)r * S * S;
  const int n = g.h * g.w;
  int nmask = 0, nbox = 0, bad = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const int y = g.b.y1 + i % g.h, x = g.b.x1 + i / g.h;
    float z;
    const bool m = roi_pixel(g, d, S, mask_s, y, x, z);
    bad |= !isfinite(z);
    nbox += z > 0.f;
    nmask += m && z > 0.f;   // (depth * mask).max() > 0 (:43) holds iff this is non-zero
  }
  nmask = block_sum(nmask, red);
  nbox = block_sum(nbox, red);
  bad = block_sum(bad, red);
  if (threadIdx.x == 0) count[r] = bad ? -2 : (nmask > 0 ? nmask : nbox);
}

// One CTA per ROI.  ranks [R,P]: indices into the ROI's valid points in column-major order (idisp_roi_points_choice).
// When count[r] equals the box area every box pixel is a point (the mask covers the whole box, or misses it and the box is kept),
// and rank c is pixel (y1 + c % h, x1 + c / h).  Otherwise the box is walked in column-major chunks of blockDim pixels: a block-wide
// exclusive scan of the mask bits ranks the chunk's points, their pixels are compacted to shared memory, and every slot whose rank
// falls in the chunk takes its pixel.  A slot whose rank is outside [0, count[r]) -- or every slot of a ROI with count[r] <= 0 --
// gets NaN coordinates and pixel -1.
__global__ void __launch_bounds__(PTS_THREADS) roi_points_gather_kernel(
    const float *__restrict__ disp, int S, const float *__restrict__ probs, int M, int pad, float thr, const float *__restrict__ lb,
    const float *__restrict__ rb, const int *__restrict__ image_index, const int *__restrict__ image_wh, const double *__restrict__ calib,
    int n_images, const int *__restrict__ count, const int *__restrict__ ranks, int P, float max_depth, float *__restrict__ pts,
    float *__restrict__ pts_mean, double *__restrict__ rot_angle, int *__restrict__ pixels)
{
  extern __shared__ float smem[];
  __shared__ int wsum[PTS_THREADS / 32];
  __shared__ float red[PTS_THREADS / 32];
  __shared__ int s_max;
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const RoiPts g = roi_pts_setup(lb, rb, r, image_index, image_wh, calib, n_images, M, pad, thr);
  float *mask_s = smem;
  int *rank_s = reinterpret_cast<int *>(mask_s + g.Mp * g.Mp);
  int *pix_s = rank_s + P;        // chosen pixel of each slot, as a column-major index into the box (-1: none)
  int *list_s = pix_s + P;        // the current chunk's compacted points
  const int n = count[r], area = g.h * g.w;
  const bool ok = !g.status && n > 0;
  if (tid == 0) s_max = -1;
  __syncthreads();
  int my_max = -1;
  for (int s = tid; s < P; s += blockDim.x) {
    const int c = ranks[(long long)r * P + s];
    const bool in = ok && c >= 0 && c < n;
    rank_s[s] = in ? c : -1;
    pix_s[s] = in && n == area ? c : -1;
    my_max = max(my_max, in ? c : -1);
  }
  if (ok) stage_mask(mask_s, probs + (long long)r * M * M, M, pad, g.Mp);
  if (ok && n != area) {
    atomicMax(&s_max, my_max);
    __syncthreads();
    const int last = s_max;
    const float *d = disp + (long long)r * S * S;
    for (int base = 0, seen = 0; base < area && seen <= last; base += blockDim.x) {   // seen, last: block-uniform
      const int i = base + tid;
      bool v = false;
      if (i < area) {
        float z;
        v = roi_pixel(g, d, S, mask_s, g.b.y1 + i % g.h, g.b.x1 + i / g.h, z) && z > 0.f;
      }
      const unsigned bal = __ballot_sync(0xffffffffu, v);
      if (lane == 0) wsum[warp] = __popc(bal);
      __syncthreads();
      int before = 0, total = 0;
      for (int k = 0; k < nw; ++k) { before += k < warp ? wsum[k] : 0; total += wsum[k]; }
      if (v) list_s[before + __popc(bal & ((1u << lane) - 1u))] = i;
      __syncthreads();
      for (int s = tid; s < P; s += blockDim.x) {
        const int c = rank_s[s] - seen;
        if (c >= 0 && c < total) pix_s[s] = list_s[c];
      }
      seen += total;
      __syncthreads();   // list_s and wsum are rewritten by the next chunk
    }
  }
  __syncthreads();
  // the points (calib.py:103-122 img_to_rect, fp32 scalars), z clamp (:84), rotation (utils_3d.py:74-104)
  const double *cal = calib + g.img * CAL_N;
  const float fu = (float)cal[CAL_FU], fv = (float)cal[CAL_FV], cu = (float)cal[CAL_CU], cv = (float)cal[CAL_CV];
  const float tx = (float)cal[CAL_TX], ty = (float)cal[CAL_TY];
  // rot_angle = atan2((x1 + x2) / 2 - W0 / 2, fu) in float64 from a float32 difference; W0: the batch's FIRST image (utils_3d.py:88)
  const float cx = __fmul_rn(__fadd_rn(lb[r * 4 + 0], lb[r * 4 + 2]), 0.5f);
  const double ang = atan2((double)__fsub_rn(cx, __fmul_rn((float)image_wh[0], 0.5f)), cal[CAL_FU]);
  const float c = (float)cos(ang), sn = (float)sin(ang);
  const float *d = disp + (long long)r * S * S;
  float sx = 0.f, sy = 0.f, sz = 0.f;
  for (int s = tid; s < P; s += blockDim.x) {
    const int i = pix_s[s];
    float px = __int_as_float(0x7fc00000), py = px, pz = px;
    if (i >= 0) {
      const int y = g.b.y1 + i % g.h, x = g.b.x1 + i / g.h;
      float z;
      roi_pixel(g, d, S, mask_s, y, x, z);
      const float X = __fadd_rn(__fdiv_rn(__fmul_rn(__fsub_rn((float)x, cu), z), fu), tx);
      const float Y = __fadd_rn(__fdiv_rn(__fmul_rn(__fsub_rn((float)y, cv), z), fv), ty);
      const float Z = fminf(z, max_depth);
      px = __fsub_rn(__fmul_rn(X, c), __fmul_rn(Z, sn));   // [x, z] @ [[c, s], [-s, c]]
      py = Y;
      pz = __fadd_rn(__fmul_rn(X, sn), __fmul_rn(Z, c));
      if (pixels) pixels[(long long)r * P + s] = y * g.W + x;
    } else if (pixels) {
      pixels[(long long)r * P + s] = -1;
    }
    float *o = pts + ((long long)r * P + s) * 3;
    o[0] = px; o[1] = py; o[2] = pz;
    sx += px; sy += py; sz += pz;
  }
  sx = block_sum(sx, red);
  sy = block_sum(sy, red);
  sz = block_sum(sz, red);
  const float mx = __fdiv_rn(sx, (float)P), my = __fdiv_rn(sy, (float)P), mz = __fdiv_rn(sz, (float)P);
  for (int s = tid; s < P; s += blockDim.x) {
    float *o = pts + ((long long)r * P + s) * 3;
    o[0] = __fsub_rn(o[0], mx); o[1] = __fsub_rn(o[1], my); o[2] = __fsub_rn(o[2], mz);
  }
  if (tid == 0) {
    pts_mean[r * 3 + 0] = mx; pts_mean[r * 3 + 1] = my; pts_mean[r * 3 + 2] = mz;
    rot_angle[r] = ang;
  }
}

// MT19937 (numpy's legacy RandomState bit generator; init_genrand seeding as np.random.seed(int) does)
struct Mt19937 {
  uint32_t mt[624];
  int pos;
  explicit Mt19937(uint32_t seed)
  {
    mt[0] = seed;
    for (int i = 1; i < 624; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    pos = 624;
  }
  uint32_t next()
  {
    if (pos >= 624) {
      for (int i = 0; i < 624; ++i) {
        const uint32_t y = (mt[i] & 0x80000000u) | (mt[(i + 1) % 624] & 0x7fffffffu);
        mt[i] = mt[(i + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
      pos = 0;
    }
    uint32_t y = mt[pos++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
  }
  // uniform in [0, max]: numpy's random_interval and its masked bounded draw (randint) -- mask = max with its bits smeared right,
  // redraw until the masked value is <= max; no draw at all for max == 0
  uint32_t interval(uint32_t max)
  {
    if (max == 0) return 0;
    uint32_t m = max;
    m |= m >> 1; m |= m >> 2; m |= m >> 4; m |= m >> 8; m |= m >> 16;
    uint32_t v;
    while ((v = next() & m) > max) {}
    return v;
  }
};

// np.random.shuffle of a 1-d array: Fisher-Yates from the end
static void shuffle_from_end(Mt19937 &g, int *a, int n)
{
  for (int i = n - 1; i >= 1; --i) std::swap(a[i], a[g.interval((uint32_t)i)]);
}

}  // namespace idisp

using namespace idisp;

static int roi_points_check(const char *who, int R, int S, int M, int n_images, float thr, int pad)
{
  IDISP_REQUIRE(R >= 0 && S > 0 && M > 0, "%s: bad shape R=%d S=%d M=%d", who, R, S, M);
  IDISP_REQUIRE(pad >= 1 && M + 2 * pad <= PTS_MAX_MASK, "%s: mask padding %d must be >= 1 and M + 2 * padding <= %d (M=%d)", who, pad,
                PTS_MAX_MASK, M);
  IDISP_REQUIRE(thr >= 0.f && thr < 1e30f, "%s: mask threshold must be finite and >= 0 (got %g)", who, (double)thr);
  IDISP_REQUIRE(R == 0 || n_images > 0, "%s: n_images must be positive", who);
  return IDISP_OK;
}

static size_t mask_smem(int M, int pad) { return sizeof(float) * (size_t)(M + 2 * pad) * (M + 2 * pad); }

extern "C" int idisp_roi_points_count(const float *roi_disp, int R, int S, const float *mask_probs, int M, const float *left_boxes,
                                      const float *right_boxes, const int *image_index, const int *image_wh, const double *calib,
                                      int n_images, float mask_threshold, int mask_padding, int *count, void *stream)
{
  int rc = roi_points_check("roi_points_count", R, S, M, n_images, mask_threshold, mask_padding);
  if (rc) return rc;
  if (R == 0) return IDISP_OK;
  IDISP_REQUIRE(roi_disp && mask_probs && left_boxes && right_boxes && image_index && image_wh && calib && count,
                "roi_points_count: NULL pointer");
  roi_points_count_kernel<<<R, PTS_THREADS, mask_smem(M, mask_padding), (cudaStream_t)stream>>>(
      roi_disp, S, mask_probs, M, mask_padding, mask_threshold, left_boxes, right_boxes, image_index, image_wh, calib, n_images, count);
  IDISP_LAUNCH_CHECK();
  return IDISP_OK;
}

extern "C" int idisp_roi_points_choice(int n, int npoints, int *out)
{
  IDISP_REQUIRE(n > 0 && npoints > 0, "roi_points_choice: n=%d and npoints=%d must be positive", n, npoints);
  IDISP_REQUIRE(out, "roi_points_choice: NULL pointer");
  const int P = npoints;
  if (n > P) {   // np.random.seed(0); choice(n, P, replace=False) = permutation(n)[:P]
    std::vector<int> perm(n);
    std::iota(perm.begin(), perm.end(), 0);
    Mt19937 g(0);
    shuffle_from_end(g, perm.data(), n);
    std::copy(perm.begin(), perm.begin() + P, out);
  } else {       // np.random.seed(0); concatenate((arange(n), choice(n, P - n, replace=True)))
    std::iota(out, out + n, 0);
    Mt19937 g(0);
    for (int i = n; i < P; ++i) out[i] = (int)g.interval((uint32_t)(n - 1));
  }
  Mt19937 g(0);  // np.random.seed(0); shuffle(choice)
  shuffle_from_end(g, out, P);
  return IDISP_OK;
}

extern "C" int idisp_roi_points_gather(const float *roi_disp, int R, int S, const float *mask_probs, int M, const float *left_boxes,
                                       const float *right_boxes, const int *image_index, const int *image_wh, const double *calib,
                                       int n_images, float mask_threshold, int mask_padding, const int *count, const int *ranks,
                                       int npoints, float max_depth, float *pts, float *pts_mean, double *rot_angle, int *pixels,
                                       void *stream)
{
  int rc = roi_points_check("roi_points_gather", R, S, M, n_images, mask_threshold, mask_padding);
  if (rc) return rc;
  IDISP_REQUIRE(npoints > 0 && npoints <= PTS_MAX_POINTS, "roi_points_gather: npoints=%d must be in [1, %d]", npoints, PTS_MAX_POINTS);
  IDISP_REQUIRE(R <= 2147483647 / npoints, "roi_points_gather: R * npoints overflows");
  IDISP_REQUIRE(!(max_depth != max_depth), "roi_points_gather: max_depth is NaN");
  if (R == 0) return IDISP_OK;
  IDISP_REQUIRE(roi_disp && mask_probs && left_boxes && right_boxes && image_index && image_wh && calib && count && ranks && pts &&
                pts_mean && rot_angle, "roi_points_gather: NULL pointer");
  const size_t smem = mask_smem(M, mask_padding) + sizeof(int) * (2 * (size_t)npoints + PTS_THREADS);
  if (smem > 48 * 1024)
    IDISP_CUDA(cudaFuncSetAttribute(roi_points_gather_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  roi_points_gather_kernel<<<R, PTS_THREADS, smem, (cudaStream_t)stream>>>(
      roi_disp, S, mask_probs, M, mask_padding, mask_threshold, left_boxes, right_boxes, image_index, image_wh, calib, n_images, count,
      ranks, npoints, max_depth, pts, pts_mean, rot_angle, pixels);
  IDISP_LAUNCH_CHECK();
  return IDISP_OK;
}
