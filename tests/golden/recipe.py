"""Deterministic recipes for test inputs and weights (shared by the golden generator and the tests).

Nothing here touches the reference or the oracle: tensors are pure functions of
(shape, seed) through ``torch.Generator`` on the CPU, so the GPU box regenerates exactly
what the authoring container used.  Every golden file also stores a checksum of each
regenerated tensor; a mismatch fails the test loudly instead of comparing garbage.
"""
import math
import zlib

import numpy as np
import torch


def _gen(seed, key):
    g = torch.Generator()
    g.manual_seed((seed * 1000003 + zlib.crc32(key.encode())) & 0x7FFFFFFF)
    return g


def make_state_dict(shapes, seed, classif_damp=0.1, raw=False):
    """shapes: {state_dict key: shape}.  'Trained-like' weights (SURVEY.md 7.3-H1):

    He-normal conv kernels, BN affine parameters jittered around (1, 0), identity BN
    running statistics (the generator calibrates them and stores the calibrated values),
    final classifier kernels damped so the soft-argmin is smooth.

    raw=True: the reference's DEFAULT INITIALISATION instead (stackhourglass.py:90-104) -- He-normal Conv2d/Conv3d kernels,
    PyTorch's own kaiming-uniform(a=sqrt(5)) for the transposed convs the init loop skips, BN (1, 0) with identity running
    statistics, nothing damped, nothing calibrated (SURVEY.md section 8c: the raw fixture next to the trained-like one).
    """
    sd = {}
    for key in sorted(shapes):
        shape = tuple(shapes[key])
        g = _gen(seed, key)
        if raw and not key.endswith('num_batches_tracked') and not key.endswith('running_mean') and not key.endswith('running_var'):
            if len(shape) >= 4:
                ksz = int(np.prod(shape[2:]))
                if ('.conv5.' in key) or ('.conv6.' in key):   # ConvTranspose3d [Cin,Cout,k,k,k]: fan_in = size(1)*k^3
                    bound = 1.0 / math.sqrt(shape[1] * ksz)
                    sd[key] = (torch.rand(shape, generator=g) * 2 - 1) * bound
                else:
                    sd[key] = torch.randn(shape, generator=g) * math.sqrt(2.0 / (ksz * shape[0]))
            else:
                sd[key] = torch.ones(shape) if key.endswith('.weight') else torch.zeros(shape)
            continue
        if key.endswith('num_batches_tracked'):
            t = torch.zeros(shape, dtype=torch.int64)
        elif key.endswith('running_mean'):
            t = torch.zeros(shape)
        elif key.endswith('running_var'):
            t = torch.ones(shape)
        elif len(shape) >= 4:  # conv / deconv kernel
            ksz = int(np.prod(shape[2:]))
            transposed = ('.conv5.' in key) or ('.conv6.' in key)
            cout = shape[1] if transposed else shape[0]
            t = torch.randn(shape, generator=g) * math.sqrt(2.0 / (ksz * cout))
            if key.startswith('classif') and key.endswith('.2.weight'):
                t = t * classif_damp
        elif key.endswith('.weight'):  # BN gamma
            t = 0.8 + 0.4 * torch.rand(shape, generator=g)
        elif key.endswith('.bias'):  # BN beta
            t = 0.05 * torch.randn(shape, generator=g)
        else:
            raise KeyError(key)
        sd[key] = t
    return sd


def make_features(B, C, Hf, Wf, seed, relu=True):
    gl, gr = _gen(seed, 'left'), _gen(seed, 'right')
    L = torch.randn(B, C, Hf, Wf, generator=gl)
    R = torch.randn(B, C, Hf, Wf, generator=gr)
    if relu:
        L, R = L.relu(), R.relu()
    return L.contiguous(), R.contiguous()


def make_stereo_crops(R, size, seed, max_shift=12):
    """R left/right ROI crop pairs [R,3,size,size] as DispRCNN3D hands them to PSMNet (disprcnn3d.py:44-50: ROIAlign-ed image
    crops, ImageNet-normalised): a smooth random texture per ROI, the right view = the left one shifted by a per-ROI number of
    pixels plus a little independent noise, so the network sees a real correspondence problem."""
    g = _gen(seed, 'crops')
    pad = 2 * max_shift
    Hb, Wb = size + 8, size + pad + 8
    noise_src = torch.rand(R, 3, Hb + 8, Wb + 8, generator=g)

    def box_blur(x, k):   # explicit shifted adds in a fixed order: bit-reproducible on any CPU (a pooling kernel's summation order is not)
        acc = torch.zeros(R, 3, Hb, Wb)
        o = 4 - k // 2
        for dy in range(k):
            for dx in range(k):
                acc = acc + x[:, :, o + dy:o + dy + Hb, o + dx:o + dx + Wb]
        return acc / float(k * k)
    base = box_blur(noise_src, 5) * 0.6 + box_blur(noise_src, 9) * 0.4
    base = (base - 0.5) * 2.5 + 0.45   # fixed affine stretch (no data-dependent statistics)
    noise = torch.randn(R, 3, size, size, generator=g) * 0.01
    shifts = torch.randint(-max_shift, max_shift + 1, (R,), generator=g)
    left = torch.stack([base[r, :, 4:4 + size, 4 + max_shift:4 + max_shift + size] for r in range(R)])
    right = torch.stack([base[r, :, 4:4 + size, 4 + max_shift + int(shifts[r]):4 + max_shift + int(shifts[r]) + size] for r in range(R)]) + noise
    mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
    return ((left.clamp(0, 1) - mean) / std).contiguous(), ((right.clamp(0, 1) - mean) / std).contiguous()


def make_images(B, H, W, seed):
    g = _gen(seed, 'images')
    return torch.rand(B, 3, H, W, generator=g).contiguous()


def checksum(t):
    a = np.ascontiguousarray(t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t)
    return np.array([zlib.crc32(a.tobytes())], dtype=np.int64)


# 3-D stack layer table: state_dict prefix -> (kind, cin, cout); cin of the first layer is 2C.
def stack3d_shapes(C):
    shapes = {}

    def convbn(p, cin, cout, transposed=False):
        shapes[p + '.0.weight'] = (cin, cout, 3, 3, 3) if transposed else (cout, cin, 3, 3, 3)
        for k in ('weight', 'bias', 'running_mean', 'running_var'):
            shapes[p + '.1.' + k] = (cout,)
        shapes[p + '.1.num_batches_tracked'] = ()

    convbn('dres0.0', 2 * C, 32)
    convbn('dres0.2', 32, 32)
    convbn('dres1.0', 32, 32)
    convbn('dres1.2', 32, 32)
    for h in ('dres2', 'dres3', 'dres4'):
        convbn(h + '.conv1.0', 32, 64)
        convbn(h + '.conv2', 64, 64)
        convbn(h + '.conv3.0', 64, 64)
        convbn(h + '.conv4.0', 64, 64)
        convbn(h + '.conv5', 64, 64, True)
        convbn(h + '.conv6', 64, 32, True)
    for c in ('classif1', 'classif2', 'classif3'):
        convbn(c + '.0', 32, 32)
        shapes[c + '.2.weight'] = (1, 32, 3, 3, 3)
    return shapes


def feature2d_shapes(prefix='feature_extraction.'):
    """state_dict keys -> shapes of the 2-D extractor (disprcnn/modeling/psmnet/submodule.py:60-110), written out by hand so
    the GPU box regenerates the weights without the reference: firstconv (3 convbn), layer1 3 x / layer2 16 x / layer3 3 x /
    layer4 3 x BasicBlock (conv1 = convbn+ReLU, conv2 = convbn, 1x1 downsample at layer2.0 and layer3.0), four SPP branches
    (1x1 convbn 128->32), lastconv (convbn 320->128 3x3, Conv2d 128->32 1x1)."""
    shapes = {}

    def bn(p, c):
        for k in ('weight', 'bias', 'running_mean', 'running_var'):
            shapes[p + '.' + k] = (c,)
        shapes[p + '.num_batches_tracked'] = ()

    def convbn(p, cin, cout, k):
        shapes[p + '.0.weight'] = (cout, cin, k, k)
        bn(p + '.1', cout)

    convbn(prefix + 'firstconv.0', 3, 32, 3)
    convbn(prefix + 'firstconv.2', 32, 32, 3)
    convbn(prefix + 'firstconv.4', 32, 32, 3)
    inpl = 32
    for name, planes, blocks, stride in (('layer1', 32, 3, 1), ('layer2', 64, 16, 2), ('layer3', 128, 3, 1), ('layer4', 128, 3, 1)):
        for b in range(blocks):
            p = f'{prefix}{name}.{b}'
            convbn(p + '.conv1.0', inpl if b == 0 else planes, planes, 3)
            convbn(p + '.conv2', planes, planes, 3)
            if b == 0 and (stride != 1 or inpl != planes):
                shapes[p + '.downsample.0.weight'] = (planes, inpl, 1, 1)
                bn(p + '.downsample.1', planes)
        inpl = planes
    for br in ('branch1', 'branch2', 'branch3', 'branch4'):
        convbn(f'{prefix}{br}.1', 128, 32, 1)
    convbn(prefix + 'lastconv.0', 320, 128, 3)
    shapes[prefix + 'lastconv.2.weight'] = (32, 128, 1, 1)
    return shapes


# whole-PSMNet cases (image crops through the real feature_extraction + the 3-D stack): the live drop-in call
# DispRCNN3D._forward_eval makes (disprcnn3d.py:266-284 -> stackhourglass.py:106-174)
PSM_CASES = {
    'psm_live': dict(R=2, size=224, mindisp=-48, maxdisp=48, seed=41),
}

# default-initialisation cases (no calibration, nothing damped): stackhourglass.py:90-104 as is
RAW_CASES = {
    'raw_tiny': dict(B=2, C=32, Hf=16, Wf=16, mindisp=-16, maxdisp=16, seed=51),
    'raw_live': dict(B=1, C=32, Hf=56, Wf=56, mindisp=-48, maxdisp=48, seed=52),
}

CASES = {
    # name: B, C, Hf, Wf, mindisp, maxdisp, seed
    'tiny': dict(B=2, C=32, Hf=16, Wf=16, mindisp=-16, maxdisp=16, seed=11),
    'tiny_pos': dict(B=1, C=32, Hf=12, Wf=20, mindisp=0, maxdisp=32, seed=12),
    'c1': dict(B=1, C=16, Hf=64, Wf=64, mindisp=-48, maxdisp=48, seed=13),
    # the shape tools/test_net.py really runs (KITTI configs: 224x224 crops -> 56x56x32ch features, D=24 -> 224x224), 2 ROI pairs
    'live': dict(B=2, C=32, Hf=56, Wf=56, mindisp=-48, maxdisp=48, seed=15),
    # one ROI pair of BASELINE.json configs[1] (the benchmark shape): 112x112x32ch, D=48 -> 448x448
    'full': dict(B=1, C=32, Hf=112, Wf=112, mindisp=-96, maxdisp=96, seed=14),
}

ROI_CASES = {
    # name: (N, C, H, W, pooled_h, pooled_w, spatial_scale, sampling_ratio, rois)
    'kitti_int': dict(N=2, C=3, H=94, W=310, ph=56, pw=56, scale=1.0, sr=0, seed=21, rois=[
        [0, 10, 5, 66, 61], [0, 100, 20, 290, 93], [1, 0, 0, 309, 93], [1, 200, 40, 256, 68],
        [0, 30, 10, 30 + 224, 10 + 80], [1, 5, 60, 12, 70]]),
    'frac_sr2': dict(N=2, C=8, H=50, W=76, ph=7, pw=7, scale=0.25, sr=2, seed=22, rois=[
        [0, 12.3, 7.9, 180.2, 150.5], [1, 0.0, 0.0, 303.9, 199.9], [0, 250.1, 100.7, 320.0, 220.0],
        [1, 40.0, 40.0, 40.4, 40.2], [0, -20.5, -9.0, 60.0, 50.0]]),
    'border': dict(N=1, C=4, H=33, W=47, ph=14, pw=9, scale=0.5, sr=0, seed=23, rois=[
        [0, 0, 0, 93, 65], [0, 80, 50, 120, 90], [0, 92, 64, 94, 66], [0, -10, -10, 4, 4]]),
}

# fresh random boxes over one input, pooled at several (pooled_h, pooled_w, spatial_scale, sampling_ratio)
ROI_RANDOM_CONFIGS = [(7, 7, 1.0, 0), (5, 9, 0.5, 2), (16, 16, 1.0, 3)]


def make_random_roi_inputs():
    """[2,5,40,60] input and 12 random boxes (some reach past the border), for golden roialign_random.npz."""
    g = torch.Generator().manual_seed(5)
    inp = torch.randn(2, 5, 40, 60, generator=g)
    xy = torch.rand(12, 2, generator=g) * torch.tensor([50., 30.])
    wh = torch.rand(12, 2, generator=g) * torch.tensor([40., 30.])
    rois = torch.cat([torch.randint(0, 2, (12, 1), generator=g).float(), xy, xy + wh], 1)
    return inp, rois


# per-ROI disparity hand-off (disprcnn3d.py:161-190, point_rcnn.py:113-136): integer-expanded boxes inside the image (the
# detector clips its boxes, structures/bounding_box.py clip_to_image), S x S ROI maps, binary masks, fu*baseline per ROI
PASTE_CASES = {
    'paste_small': dict(H=96, W=310, S=32, seed=61, boxes=[
        # per image: (left box, right box)
        [([10.3, 5.2, 70.8, 60.1], [2.1, 5.2, 60.0, 60.1]), ([100.0, 20.0, 289.5, 92.7], [80.4, 20.0, 275.0, 92.7]),
         ([40.2, 30.9, 120.4, 80.0], [30.0, 30.9, 118.9, 80.0])],
        [([0.0, 0.0, 309.0, 95.0], [0.0, 0.0, 300.2, 95.0]), ([200.6, 40.1, 256.3, 68.8], [190.2, 40.1, 250.0, 68.8])],
        [],
    ]),
}


def make_paste_inputs(case):
    g = _gen(case['seed'], 'paste')
    lbs = [[list(b[0]) for b in img] for img in case['boxes']]
    rbs = [[list(b[1]) for b in img] for img in case['boxes']]
    R = sum(len(i) for i in lbs)
    disp = (torch.randn(R, case['S'], case['S'], generator=g) * 6.0 + 4.0).contiguous()
    masks = (torch.rand(R, case['H'], case['W'], generator=g) > 0.3).to(torch.uint8).contiguous()
    fub = (300.0 + 200.0 * torch.rand(R, generator=g)).contiguous()
    return disp, lbs, rbs, masks, fub
