"""Deterministic inputs for the per-ROI point-cloud hand-off (PointRCNN.process_input_eval, point_rcnn.py:189-242).

Like recipe.py: pure functions of (case, seed) through ``torch.Generator`` on the CPU, so the GPU box regenerates exactly what the
golden generator fed the reference; the fixture stores checksums of the regenerated tensors.
"""
import numpy as np
import torch

import recipe

# Two KITTI-sized images with distinct, KITTI-like P2 / P3 (3x4, float64).  Per ROI: (left box, right box, mask kind, disparity
# mean, disparity std).  The ROIs cover: n > 768 (a large box), n < 768 (a small box under a sparse mask), n == 768 exactly (a 32 x 24
# box whose mask misses it -> the unmasked fallback), masks reaching past the integer box, a box on the image border, disparities
# that clamp z at 160 (tiny disparities) and depth at 1 (a right box 410 px to the left).
POINTS_CASES = {
    'points_kitti': dict(S=224, M=28, npoints=768, seed=71, images=[
        dict(size=(1242, 375),
             P2=[[721.5377, 0.0, 609.5593, 44.85728], [0.0, 721.5377, 172.854, 0.2163791], [0.0, 0.0, 1.0, 0.002745884]],
             P3=[[721.5377, 0.0, 609.5593, -339.5242], [0.0, 721.5377, 172.854, 2.199936], [0.0, 0.0, 1.0, 0.002729905]],
             rois=[([400.3, 150.7, 620.2, 300.4], [360.1, 150.7, 585.6, 300.4], 'blob', 38.0, 3.0),
                   ([100.5, 180.2, 130.8, 205.9], [80.2, 180.2, 111.0, 205.9], 'sparse', 20.0, 2.0),
                   ([700.0, 200.0, 732.0, 224.0], [690.0, 200.0, 722.0, 224.0], 'low', 9.0, 1.5),
                   ([850.6, 120.3, 950.2, 220.8], [825.0, 120.3, 930.4, 220.8], 'full', 24.0, 2.0),
                   ([1180.4, 300.2, 1242.0, 375.0], [1150.2, 300.2, 1230.5, 375.0], 'blob', 30.0, 2.5)]),
        dict(size=(1224, 375),
             P2=[[707.0493, 0.0, 604.0814, 45.75831], [0.0, 707.0493, 180.5066, -0.3454157], [0.0, 0.0, 1.0, 0.004981016]],
             P3=[[707.0493, 0.0, 604.0814, -334.1081], [0.0, 707.0493, 180.5066, 0.3330294], [0.0, 0.0, 1.0, 0.003201153]],
             rois=[([600.2, 100.1, 680.7, 160.3], [190.5, 100.1, 275.0, 160.3], 'blob', 0.0, 4.0),
                   ([300.5, 180.6, 360.2, 230.1], [299.8, 180.6, 359.0, 230.1], 'full', 0.3, 0.3),
                   ([0.0, 40.4, 210.9, 190.6], [0.0, 40.4, 190.2, 190.6], 'blob', 15.0, 4.0)]),
    ]),
}


def mask_probs(kind, M, g):
    """[M,M] mask probabilities: 'blob' (a smooth object), 'sparse' (a few isolated confident cells), 'low' (nothing above 0.5),
    'full' (confident everywhere, so the pasted mask reaches past the integer box)."""
    if kind == 'low':
        return 0.05 + 0.35 * torch.rand(M, M, generator=g)
    if kind == 'full':
        return 0.8 + 0.19 * torch.rand(M, M, generator=g)
    if kind == 'sparse':
        p = 0.3 * torch.rand(M, M, generator=g)
        keep = torch.rand(M, M, generator=g) < 0.08
        return torch.where(keep, 0.75 + 0.2 * torch.rand(M, M, generator=g), p)
    yy, xx = torch.meshgrid(torch.linspace(-1, 1, M), torch.linspace(-1, 1, M), indexing='ij')
    field = 2.5 * (1.0 - (xx / 0.8) ** 2 - (yy / 0.9) ** 2) + 0.8 * torch.randn(M, M, generator=g)
    return torch.sigmoid(field)


def make_points_inputs(case, seed):
    """roi_disp [R,S,S] f32, mask_probs [R,1,M,M] f32, left / right boxes [R,4] f32, rois_per_image, P2 / P3 per image."""
    g = recipe._gen(seed, 'points')
    S, M = case['S'], case['M']
    disp, probs, lbs, rbs, counts = [], [], [], [], []
    for img in case['images']:
        counts.append(len(img['rois']))
        for lb, rb, kind, mean, std in img['rois']:
            lo = torch.randn(1, 1, S // 16, S // 16, generator=g)
            smooth = torch.nn.functional.interpolate(lo, (S, S), mode='bilinear', align_corners=True)[0, 0]
            disp.append(mean + std * (0.7 * smooth + 0.3 * torch.randn(S, S, generator=g)))
            probs.append(mask_probs(kind, M, g)[None])
            lbs.append(lb)
            rbs.append(rb)
    return (torch.stack(disp).contiguous().float(), torch.stack(probs).contiguous().float(), torch.tensor(lbs, dtype=torch.float32),
            torch.tensor(rbs, dtype=torch.float32), counts, [np.asarray(i['P2']) for i in case['images']],
            [np.asarray(i['P3']) for i in case['images']])


def checksums(disp, probs, lb, rb):
    return np.array([int(recipe.checksum(t)[0]) for t in (disp, probs, lb, rb)], dtype=np.int64)


def make_kitti_batch(R_per_image, seed, S=224, M=28, W=1242, H=375):
    """A seeded KITTI-size batch of random ROIs: image i gets R_per_image[i] boxes (fully inside the image, 24..220 px wide, right
    box shifted left by 5..60 px), 'blob' masks and disparities around the box's shift.  Same P2 / P3 for every image."""
    g = recipe._gen(seed, 'points_batch')
    base = POINTS_CASES['points_kitti']['images'][0]
    disp, probs, lbs, rbs = [], [], [], []
    for _ in range(sum(R_per_image)):
        w = 24 + 196 * float(torch.rand((), generator=g))
        h = 20 + 130 * float(torch.rand((), generator=g))
        x1 = 1 + (W - w - 2) * float(torch.rand((), generator=g))
        y1 = 1 + (H - h - 2) * float(torch.rand((), generator=g))
        sh = 5 + 55 * float(torch.rand((), generator=g))
        lbs.append([x1, y1, x1 + w, y1 + h])
        rbs.append([max(x1 - sh, 0.0), y1, max(x1 - sh, 0.0) + w * 0.95, y1 + h])
        lo = torch.randn(1, 1, S // 16, S // 16, generator=g)
        smooth = torch.nn.functional.interpolate(lo, (S, S), mode='bilinear', align_corners=True)[0, 0]
        disp.append(2.0 + 3.0 * smooth + 0.5 * torch.randn(S, S, generator=g))
        probs.append(mask_probs('blob', M, g)[None])
    n = len(R_per_image)
    return (torch.stack(disp).float() if disp else torch.zeros(0, S, S), torch.stack(probs).float() if probs else torch.zeros(0, 1, M, M),
            torch.tensor(lbs, dtype=torch.float32).reshape(-1, 4), torch.tensor(rbs, dtype=torch.float32).reshape(-1, 4), list(R_per_image),
            [np.asarray(base['P2'])] * n, [np.asarray(base['P3'])] * n, [(W, H)] * n)
