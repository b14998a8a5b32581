"""Oracle of the per-ROI point-cloud hand-off -- TEST INFRASTRUCTURE ONLY (the product never imports it).

A torch restatement, device-agnostic, of PointRCNN.process_input_eval + back_project(fix_seed=True)
(disprcnn/modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:189-242, :37-85) on flat inputs, shaped like the reference:
per ROI an image-sized depth map, the Masker's image-sized mask, depthmap_to_rect over every pixel, nonzero, numpy's seeded
sampling.  Same arguments and results as ``disprcnn_b200.layers.roi_points`` (so tools/bench_points.py times it as the
reference-shaped baseline on the GPU), except that it also returns the chosen pixels and the per-ROI counts.
"""
import numpy as np
import torch
import torch.nn.functional as F

import idispnet_oracle as O


def paste_mask(mask, box, im_h, im_w, thresh=0.5, padding=1):
    """Masker.forward_single_image for one ROI (modeling/roi_heads/mask_head/inference.py:91-159): mask [M,M] probabilities, box [4]
    float32 -> [im_h, im_w] uint8."""
    mask, box = mask.float(), box.float()
    M = mask.shape[-1]
    scale = float(M + 2 * padding) / M                                       # expand_masks, :109-118
    padded = mask.new_zeros((M + 2 * padding, M + 2 * padding))
    padded[padding:-padding, padding:-padding] = mask
    w_half, h_half = (box[2] - box[0]) * .5, (box[3] - box[1]) * .5          # expand_boxes, :91-106
    x_c, y_c = (box[2] + box[0]) * .5, (box[3] + box[1]) * .5
    w_half, h_half = w_half * scale, h_half * scale
    b = torch.stack([x_c - w_half, y_c - h_half, x_c + w_half, y_c + h_half]).to(dtype=torch.int32).tolist()
    w, h = max(b[2] - b[0] + 1, 1), max(b[3] - b[1] + 1, 1)
    m = F.interpolate(padded[None, None], size=(h, w), mode='bilinear', align_corners=False)[0, 0] > thresh
    im = torch.zeros((im_h, im_w), dtype=torch.uint8, device=mask.device)
    x0, x1, y0, y1 = max(b[0], 0), min(b[2] + 1, im_w), max(b[1], 0), min(b[3] + 1, im_h)
    im[y0:y1, x0:x1] = m[y0 - b[1]:y1 - b[1], x0 - b[0]:x1 - b[0]]
    return im


def choice(n, npoints):
    """back_project's sampling (point_rcnn.py:53-74) with fix_seed=True."""
    if n > npoints:
        np.random.seed(0)
        c = np.random.choice(n, npoints, replace=False)
    else:
        np.random.seed(0)
        c = np.random.choice(n, npoints - n, replace=True)
        c = np.concatenate((np.arange(n), c))
    np.random.seed(0)
    np.random.shuffle(c)
    return c


def roi_points(roi_disp, mask_probs, left_boxes, right_boxes, rois_per_image, calibs, image_sizes, npoints=768, max_depth=160.,
               mask_threshold=0.5, mask_padding=1):
    """-> pts [R,P,3], pts_mean [R,3], rot_angle [R] f64, pixels [R,P] int64 (y * width + x), counts [R] int64 (the number of valid
    points of each ROI), all on roi_disp's device.  calibs: rows (fu, fv, cu, cv, tx, ty, fu*b) per image; image_sizes (w, h)."""
    dev = roi_disp.device
    R = roi_disp.shape[0]
    M = mask_probs.shape[-1]
    probs = mask_probs.reshape(R, M, M)
    image_of = [i for i, c in enumerate(rois_per_image) for _ in range(int(c))]
    pts_list, pix_list, counts = [], [], []
    for r in range(R):
        i = image_of[r]
        W, H = (int(v) for v in image_sizes[i])
        fu, fv, cu, cv, tx, ty, fub = (float(v) for v in calibs[i])
        lb, rb = left_boxes[r].tolist(), right_boxes[r].tolist()
        d, (x1, y1, x2, y2), x1p = O._resize_crop_shift(roi_disp[r], lb, rb)   # DisparityMap resize / crop, :210-213
        d = d + x1 - x1p                                                        # :214
        depth = torch.zeros((H, W), device=dev)
        depth[y1:y2, x1:x2] = (fub / (d + 1e-6)).clamp(min=1.0)                # :215-218
        mask = paste_mask(probs[r], left_boxes[r], H, W, mask_threshold, mask_padding)
        if mask.sum() != 0 and (depth * mask.float()).max() > 0:               # back_project :42-43
            depth = depth * mask.float()
        xs, ys = torch.meshgrid(torch.arange(W, device=dev), torch.arange(H, device=dev), indexing='ij')   # calib.py:103-112
        xs, ys = xs.reshape(-1), ys.reshape(-1)
        z = depth[ys, xs]
        x = ((xs.float() - cu) * z) / fu + tx                                   # calib.py img_to_rect :95-101
        y = ((ys.float() - cv) * z) / fv + ty
        pos = torch.nonzero(z > 0).squeeze(1)                                   # :54
        if len(pos) == 0:
            raise EOFError('mask is nonvalid')
        idx = pos[torch.from_numpy(choice(len(pos), npoints)).to(dev)]
        pts_list.append(torch.stack([x[idx], y[idx], z[idx]], 1))
        pix_list.append(ys[idx] * W + xs[idx])
        counts.append(len(pos))
    if R == 0:
        e = torch.zeros((0,), device=dev)
        return (e.new_zeros((0, npoints, 3)), e.new_zeros((0, 3)), e.new_zeros((0,), dtype=torch.float64),
                e.new_zeros((0, npoints), dtype=torch.int64), e.new_zeros((0,), dtype=torch.int64))
    pts = torch.stack(pts_list)
    pts[:, :, 2] = torch.clamp(pts[:, :, 2].clone(), max=max_depth)            # :84
    # rotate_pc_along_y (utils/utils_3d.py:74-104): W0 = the first image's width; fu per ROI as float64 (torch.tensor(fus))
    fus = torch.tensor([float(calibs[i][0]) for i in image_of], dtype=torch.float64, device=dev)
    cx = (left_boxes[:, 0] + left_boxes[:, 2]) / 2
    rot_angle = torch.atan2(cx - image_sizes[0][0] / 2, fus)
    c, s = torch.cos(rot_angle).unsqueeze(1), torch.sin(rot_angle).unsqueeze(1)
    rotmat = torch.cat([c, -s, s, c], dim=1).view(-1, 2, 2)
    pts[:, :, [0, 2]] = torch.bmm(pts[:, :, [0, 2]], torch.transpose(rotmat, 1, 2).float())
    pts_mean = pts.mean(1)
    return (pts - pts_mean[:, None, :], pts_mean, rot_angle, torch.stack(pix_list),
            torch.tensor(counts, dtype=torch.int64, device=dev))

