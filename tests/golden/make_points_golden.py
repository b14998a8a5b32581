"""Generate tests/golden/points_*.npz by EXECUTING THE REFERENCE's PointRCNN.process_input_eval (authoring machine only).

Run:  python tests/golden/make_points_golden.py [points_kitti ...]
Needs a checkout of the reference project: $REFERENCE_ROOT, by default `reference` next to this repository.  GPU tests only read the .npz.

What is executed: ``PointRCNN.process_input_eval`` (disprcnn/modeling/pointnet_module/point_rcnn/lib/net/point_rcnn.py:189-242)
and ``back_project`` (:37-85) from the UNMODIFIED module, on the reference's own ``BoxList`` / ``Calib(Calibration(...))`` objects
and a stand-in ``self`` with ``cfg.RPN.NPOINTS``.  The module imports once the CUDA-only packages it names at import time
(pycocotools, pointnet2_cuda, roipool3d_cuda, iou3d_cuda -- none is called on this path) are stubbed; ``Tensor.cuda`` is the
identity for the call.  Stored: the returned ``pts``, ``self.pts_mean``, ``self.rotator.rot_angle``; the per-ROI counts and the
chosen pixels, derived from the masked depth maps ``back_project`` leaves behind and checked against ``pts`` here; the Masker's
masks (packed bits); the input checksums and the seed.  A seed whose pre-threshold mask value at some in-box pixel lies within
1e-6 of the threshold is skipped (the next one is tried), so the mask comparison can be exact.
"""
import os
import sys
import types
import warnings

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REFERENCE_ROOT = os.environ.get('REFERENCE_ROOT', os.path.join(os.path.dirname(ROOT), 'reference'))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.path.insert(0, REFERENCE_ROOT)
sys.path.insert(0, ROOT)

import points_oracle  # noqa: E402
import points_recipe  # noqa: E402


def _import_reference():
    for m in ('pycocotools', 'pycocotools.mask', 'pointnet2_cuda', 'roipool3d_cuda', 'iou3d_cuda'):
        sys.modules.setdefault(m, types.ModuleType(m))
    import disprcnn_b200
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        disprcnn_b200.install(inference_only=True)   # disprcnn._C shim: disprcnn.layers imports it
        from disprcnn.modeling.pointnet_module.point_rcnn.lib.net.point_rcnn import PointRCNN
    return PointRCNN


def _tie_free(probs, lbs, sizes_of, thresh, padding):
    """No in-box pixel's pre-threshold mask value within 1e-6 of the threshold (reference helpers, inference.py:91-118)."""
    from disprcnn.modeling.roi_heads.mask_head.inference import expand_boxes, expand_masks
    from disprcnn.utils.stereo_utils import expand_box_to_integer
    for r in range(probs.shape[0]):
        padded, scale = expand_masks(probs[r:r + 1], padding=padding)
        b = expand_boxes(lbs[r][None], scale)[0].to(dtype=torch.int32)
        w, h = max(int(b[2] - b[0] + 1), 1), max(int(b[3] - b[1] + 1), 1)
        v = F.interpolate(padded, size=(h, w), mode='bilinear', align_corners=False)[0, 0]
        W, H = sizes_of[r]
        full = torch.full((H, W), -1.0)
        x0, x1, y0, y1 = max(int(b[0]), 0), min(int(b[2]) + 1, W), max(int(b[1]), 0), min(int(b[3]) + 1, H)
        full[y0:y1, x0:x1] = v[y0 - int(b[1]):y1 - int(b[1]), x0 - int(b[0]):x1 - int(b[0])]
        bx1, by1, bx2, by2 = expand_box_to_integer(lbs[r].tolist())
        if ((full[by1:by2, bx1:bx2] - thresh).abs() < 1e-6).any():
            return False
    return True


def gen_points(name, case):
    PointRCNN = _import_reference()
    from disprcnn.modeling.roi_heads.mask_head.inference import Masker
    from disprcnn.structures.bounding_box import BoxList
    from disprcnn.structures.calib import Calib
    from disprcnn.utils.kitti_utils import Calibration
    thresh, padding, P = 0.5, 1, case['npoints']
    sizes = [img['size'] for img in case['images']]
    seed = case['seed']
    while True:
        disp, probs, lb, rb, counts, P2s, P3s = points_recipe.make_points_inputs(case, seed)
        sizes_of = [sizes[i] for i, c in enumerate(counts) for _ in range(c)]
        if _tie_free(probs, lb, sizes_of, thresh, padding):
            break
        print(f'{name}: seed {seed} has a mask value within 1e-6 of {thresh}; trying {seed + 1}')
        seed += 1
    lefts, rights, targets, r0 = [], [], [], 0
    for i, (W, H) in enumerate(sizes):
        sl = slice(r0, r0 + counts[i])
        r0 += counts[i]
        left = BoxList(lb[sl].clone(), (W, H))
        left.add_field('disparity', disp[sl].clone())
        left.add_field('mask', probs[sl].clone())
        lefts.append(left)
        rights.append(BoxList(rb[sl].clone(), (W, H)))
        eye34 = np.hstack([np.eye(3), np.zeros((3, 1))])
        cal = Calibration(dict(P0=eye34, P1=eye34, P2=P2s[i], P3=P3s[i], R0_rect=np.eye(3), Tr_velo_to_cam=eye34, Tr_imu_to_velo=eye34),
                          (W, H))
        t = BoxList(torch.zeros((0, 4)), (W, H))
        t.add_field('calib', Calib(cal, (W, H)))
        targets.append(t)
    # stand-in self: the method reads self.cfg.RPN.NPOINTS, calls self.back_project and sets self.rotator / self.pts_mean
    me = types.SimpleNamespace(cfg=types.SimpleNamespace(RPN=types.SimpleNamespace(NPOINTS=P)))
    captured = {}

    def back_project(depth_maps, mask_pred, targets, max_depth=160, fix_seed=False):
        out = PointRCNN.back_project(me, depth_maps, mask_pred, targets, max_depth=max_depth, fix_seed=fix_seed)
        captured['depth_maps'] = depth_maps   # masked in place by back_project (:42-43)
        return out
    me.back_project = back_project
    cuda = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        with torch.no_grad():
            pts = PointRCNN.process_input_eval(me, lefts, rights, targets, threshold=thresh, padding=padding)
    finally:
        torch.Tensor.cuda = cuda
    # counts and chosen pixels from the masked depth maps; rebuild pts from them with the reference's own calls
    n_all, pix_all, sel_all = [], [], []
    for i, dms in enumerate(captured['depth_maps']):
        W, H = sizes[i]
        calib = targets[i].get_field('calib')
        for dm in dms:
            zt = dm.t().reshape(-1)                       # depthmap_to_rect order: x outer, y inner (calib.py:106-108)
            pos = torch.nonzero(zt > 0).squeeze(1)
            k = pos[torch.from_numpy(points_oracle.choice(len(pos), P))]
            n_all.append(len(pos))
            pix_all.append((k % H) * W + k // H)
            sel_all.append(calib.depthmap_to_rect(dm)[0][k])
    sel = torch.stack(sel_all)
    sel[:, :, 2] = torch.clamp(sel[:, :, 2].clone(), max=160)
    n160, n1 = int((sel[:, :, 2] == 160).sum()), int((sel[:, :, 2] == 1).sum())   # (the rotator below writes into sel)
    rebuilt = me.rotator(sel.permute(0, 2, 1)).permute(0, 2, 1) - me.pts_mean[:, None, :]
    assert torch.equal(rebuilt, pts), float((rebuilt - pts).abs().max())
    masks = [Masker(threshold=thresh, padding=padding)([probs[sum(counts[:i]):sum(counts[:i + 1])]], [lefts[i]])[0][:, 0]
             for i in range(len(sizes))]
    out = dict(pts=pts.numpy(), pts_mean=me.pts_mean.numpy(), rot_angle=me.rotator.rot_angle.numpy(),
               counts=np.asarray(n_all, np.int64), pixels=torch.stack(pix_all).numpy().astype(np.int64),
               input_crc=points_recipe.checksums(disp, probs, lb, rb), seed=np.array([seed]))
    for i, m in enumerate(masks):
        out[f'masks{i}'] = np.packbits(m.numpy().astype(np.uint8).reshape(m.shape[0], -1), axis=1)
    assert out['rot_angle'].dtype == np.float64
    print(f'{name}: seed {seed}; {len(n_all)} ROIs, counts {n_all}; |pts| max {float(pts.abs().max()):.2f}; '
          f'z clamped at 160: {n160} points, depth clamped at 1: {n1}')
    np.savez_compressed(os.path.join(HERE, f'{name}.npz'), **out)


if __name__ == '__main__':
    for name in sys.argv[1:] or list(points_recipe.POINTS_CASES):
        gen_points(name, points_recipe.POINTS_CASES[name])
