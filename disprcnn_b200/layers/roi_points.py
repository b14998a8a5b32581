"""Per-ROI point clouds for PointRCNN straight from iDispNet's per-ROI disparity maps (SURVEY.md section 8(f) row 3, point-cloud half).

``roi_points`` replaces the eval-time hand-off ``PointRCNN.process_input_eval`` + ``back_project(..., fix_seed=True)``
(disprcnn/modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:189-242, :37-85): the Masker paste, the per-ROI image-sized
depth map, ``depthmap_to_rect`` over every pixel of the image, ``nonzero``, numpy's seeded sampling, the depth clamp, the rotation
about y and the centring.  Three steps on the current stream (csrc/roi_points.cu):

1. ``idisp_roi_points_count`` -- one CTA per ROI counts the ROI's points (box pixels inside the mask, or the whole box when the mask
   misses it);
2. one device-to-host copy of the R counts, then ``idisp_roi_points_choice`` per ROI on the host -- numpy's ``seed(0)``, ``choice``
   and ``shuffle`` restated bit for bit -- and one host-to-device copy of the [R, npoints] rank table;
3. ``idisp_roi_points_gather`` -- one CTA per ROI maps ranks to pixels and writes the rotated, centred points.

Nothing image-sized is allocated.  ``process_input_eval`` mirrors the reference method's signature on BoxList-like inputs.
"""
import numpy as np
import torch

from .. import _lib
from .roi_disparity import _boxes

_CODES = {-1: 'its integer box is not inside its image', -2: 'its depth is not finite inside its box (NaN or inf disparity)',
          -3: 'its image index is out of range'}


def calib_row(P2, P3):
    """(fu, fv, cu, cv, tx, ty, fu*baseline) of one image from its 3x4 P2 / P3 matrices, as the reference derives them:
    ``Calibration.fu .. ty`` in float64 (utils/kitti_utils.py:27-49) and ``Calib.stereo_fuxbaseline`` = P2[0,3] - P3[0,3] of the
    float32 copies (structures/calib.py:18-24,45-47)."""
    P2 = np.asarray(P2, dtype=np.float64).reshape(3, 4)
    P3 = np.asarray(P3, dtype=np.float64).reshape(3, 4)
    fu, fv = P2[0, 0], P2[1, 1]
    fub = np.float32(P2[0, 3]) - np.float32(P3[0, 3])
    return [fu, fv, P2[0, 2], P2[1, 2], P2[0, 3] / -fu, P2[1, 3] / -fv, float(fub)]


def roi_points(roi_disp, mask_probs, left_boxes, right_boxes, rois_per_image, calibs, image_sizes, npoints=768, max_depth=160.,
               mask_threshold=0.5, mask_padding=1, return_pixels=False):
    """Point cloud of every ROI, as ``PointRCNN.process_input_eval`` builds it.

    roi_disp [R,S,S] f32 CUDA: iDispNet's disparity per ROI; mask_probs [R,M,M] or [R,1,M,M]: the ROI's mask probabilities;
    left_boxes / right_boxes [R,4] (x1,y1,x2,y2); ROIs grouped by image, ``rois_per_image`` ROIs for each of the N images.
    calibs: N rows (fu, fv, cu, cv, tx, ty, fu*baseline) -- see ``calib_row``; image_sizes: N (width, height) pairs.

    Returns ``(pts [R,npoints,3] f32, pts_mean [R,3] f32, rot_angle [R] f64)`` and, with ``return_pixels``, ``pixels [R,npoints]``
    int32 (y * width + x of each point): ``pts`` is what the reference method returns, ``pts_mean`` and ``rot_angle`` what it keeps
    in ``self.pts_mean`` and ``self.rotator.rot_angle`` for ``rotate_back``.  Every ROI uses its own image's calib; the rotation
    angle uses the width of image 0 for every ROI, as ``rotate_pc_along_y`` does (utils/utils_3d.py:88).

    Raises ``ValueError('mask is nonvalid')`` for a ROI without points (the reference's ``EOFError``, point_rcnn.py:76) and
    ``RuntimeError`` naming the ROI when its box is not inside its image or its depth is not finite."""
    _lib.require_cuda(roi_disp, mask_probs, left_boxes, right_boxes)
    dev = roi_disp.device
    roi_disp = roi_disp.contiguous().float()
    R, S = roi_disp.shape[0], roi_disp.shape[-1]
    if roi_disp.dim() != 3 or roi_disp.shape[1] != S:
        raise RuntimeError('roi_points: roi_disp must be [R,S,S]')
    M = mask_probs.shape[-1]
    if mask_probs.numel() != R * M * M or mask_probs.shape[-2] != M:
        raise RuntimeError(f'roi_points: mask_probs {tuple(mask_probs.shape)} is not [R,M,M] or [R,1,M,M] for R={R}')
    probs = mask_probs.reshape(R, M, M).contiguous().float()
    lb, rb = _boxes(left_boxes, right_boxes)
    counts = [int(c) for c in rois_per_image]
    N = len(counts)
    if sum(counts) != R or lb.shape[0] != R:
        raise RuntimeError(f'roi_points: {R} ROI maps, {lb.shape[0]} boxes, rois_per_image sums to {sum(counts)}')
    cal = np.asarray(calibs, dtype=np.float64).reshape(-1, 7) if N else np.zeros((0, 7))
    wh = np.asarray(image_sizes, dtype=np.int64).reshape(-1, 2) if N else np.zeros((0, 2), np.int64)
    if cal.shape[0] != N or wh.shape[0] != N:
        raise RuntimeError(f'roi_points: {N} images but {cal.shape[0]} calib rows and {wh.shape[0]} image sizes')
    P = int(npoints)
    if P <= 0:
        raise ValueError(f'roi_points: npoints must be positive (got {P})')
    pts = torch.empty((R, P, 3), dtype=torch.float32, device=dev)
    pts_mean = torch.empty((R, 3), dtype=torch.float32, device=dev)
    rot_angle = torch.empty((R,), dtype=torch.float64, device=dev)
    pixels = torch.empty((R, P), dtype=torch.int32, device=dev) if return_pixels else None
    if R == 0:
        return (pts, pts_mean, rot_angle, pixels) if return_pixels else (pts, pts_mean, rot_angle)
    image_index = torch.repeat_interleave(torch.arange(N, dtype=torch.int32), torch.tensor(counts, dtype=torch.int64)).to(dev)
    image_wh = torch.from_numpy(wh.astype(np.int32)).to(dev)
    calib = torch.from_numpy(cal).to(dev)
    lib = _lib.load()
    args = (_lib.ptr(roi_disp), R, S, _lib.ptr(probs), M, _lib.ptr(lb), _lib.ptr(rb), _lib.ptr(image_index), _lib.ptr(image_wh),
            _lib.ptr(calib), N, float(mask_threshold), int(mask_padding))
    count = torch.empty((R,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.idisp_roi_points_count(*args, _lib.ptr(count), _lib.stream_ptr()))
        n = count.cpu()   # the one device-to-host copy (synchronises the current stream)
        for r, c in enumerate(n.tolist()):
            if c < 0:
                raise RuntimeError(f'roi_points: ROI {r} (image {int(image_index[r])}, box {lb[r].tolist()}): {_CODES.get(c, c)}')
            if c == 0:
                raise ValueError(f'roi_points: ROI {r}: mask is nonvalid (no point with depth > 0)')
        ranks = torch.empty((R, P), dtype=torch.int32, pin_memory=True)
        for r, c in enumerate(n.tolist()):
            _lib.check(lib.idisp_roi_points_choice(c, P, _lib.ptr(ranks[r])))
        ranks = ranks.to(dev, non_blocking=True)
        _lib.check(lib.idisp_roi_points_gather(*args, _lib.ptr(count), _lib.ptr(ranks), P, float(max_depth), _lib.ptr(pts),
                                               _lib.ptr(pts_mean), _lib.ptr(rot_angle), _lib.ptr(pixels), _lib.stream_ptr()))
    return (pts, pts_mean, rot_angle, pixels) if return_pixels else (pts, pts_mean, rot_angle)


def _p2_p3(calib):
    c = getattr(calib, 'calib', calib)   # structures/calib.py Calib wraps a kitti_utils Calibration (float64 P2 / P3)
    if isinstance(c, dict):
        return c['P2'], c['P3']
    return c.P2, c.P3


def process_input_eval(left_inputs, right_inputs, targets, threshold=0.5, padding=1, npoints=768, max_depth=160.):
    """Mirror of ``PointRCNN.process_input_eval(left_inputs, right_inputs, targets, threshold, padding)`` (point_rcnn.py:189-242) on
    BoxList-like objects: ``left_inputs[i].bbox`` [Ri,4], ``.size`` (width, height), ``.get_field('disparity')`` [Ri,S,S],
    ``.get_field('mask')`` [Ri,1,M,M]; ``right_inputs[i].bbox``; ``targets[i].get_field('calib')`` with P2 / P3 (a ``Calib``, its
    ``Calibration`` or a dict).  Returns ``(pts, pts_mean, rot_angle)``: the reference returns ``pts`` and stores the other two in
    ``self.pts_mean`` and ``self.rotator.rot_angle``.

    One deliberate difference: every ROI is back-projected with its OWN image's calib.  The reference's ``back_project`` indexes
    ``targets[i]`` by the position of the image among the images that HAVE ROIs (:232-235 -> :47-50), so an image without ROIs
    before one with ROIs shifts the later images onto the wrong calib."""
    disp, masks, lbs, rbs, counts, calibs, sizes = [], [], [], [], [], [], []
    for left, right, target in zip(left_inputs, right_inputs, targets):
        counts.append(len(left.bbox))
        sizes.append(tuple(int(v) for v in left.size))
        calibs.append(calib_row(*_p2_p3(target.get_field('calib'))))
        if len(left.bbox):
            lbs.append(left.bbox)
            rbs.append(right.bbox)
            disp.append(left.get_field('disparity'))
            masks.append(left.get_field('mask'))
    if not lbs:
        dev = torch.device('cuda', torch.cuda.current_device())
        z = torch.empty((0, 4), device=dev)
        return roi_points(torch.empty((0, 1, 1), device=dev), torch.empty((0, 1, 1), device=dev), z, z, counts, calibs, sizes, npoints,
                          max_depth, threshold, padding)
    return roi_points(torch.cat(disp), torch.cat(masks), torch.cat(lbs), torch.cat(rbs), counts, calibs, sizes, npoints, max_depth,
                      threshold, padding)
