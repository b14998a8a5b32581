"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE (authoring container only).

Run:  python tests/golden/make_golden.py
Needs /root/reference (read-only reference checkout) and, for the ROIAlign vectors,
oracle/_ref/ref_roialign.so (python oracle/build_ref.py).  The GPU box has neither; it
only consumes the committed .npz files.

What is executed:
  * iDispNet: ``disprcnn.modeling.psmnet.stackhourglass.PSMNet`` imported unmodified.
    ``PSMNet.forward`` (stackhourglass.py:106-174) runs verbatim with
    ``feature_extraction`` swapped for ``nn.Identity`` so that the inputs ARE the feature
    maps (BASELINE.json configs 1-3 are feature-input configs); a forward pre-hook on
    ``dres0`` captures the reference's own cost volume.  That "genuine" forward yields
    disparity at H,W = Hf,Wf.  The 4x-upsampled variant (H,W = 4Hf,4Wf) re-runs lines
    :130-174 on the reference's own sub-modules.
  * The same network in float64 (``.double()``) as arbiter (SURVEY.md 7.3-H1).
  * The live drop-in call (``psm_*``): ``PSMNet.forward`` UNMODIFIED -- real ``feature_extraction`` on [R,3,224,224] crop pairs
    (what ``DispRCNN3D._forward_eval`` does, disprcnn3d.py:266-284) -- plus the reference's own per-view features.
  * ``raw_*``: the 3-D stack with the reference's DEFAULT initialisation (stackhourglass.py:90-104), uncalibrated.
  * ``paste_*``: the reference's ``DisparityMap.resize / crop`` (structures/disparity.py:39-78) executed inside restatements of its two
    call-site loops (disprcnn3d.py:161-190, point_rcnn.py:113-136).
  * ROIAlign: the reference CPU kernel compiled from its own source.
BatchNorm running statistics are calibrated by two train-mode passes of the reference
and stored in the fixture (weights themselves are regenerated from tests/golden/recipe.py).
"""
import os
import sys

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)

import recipe  # noqa: E402
from disprcnn.modeling.psmnet.stackhourglass import PSMNet  # noqa: E402  (the reference)
from disprcnn.modeling.psmnet import submodule as ref_sub  # noqa: E402


def ref_tail(m, cost, H, W):
    """stackhourglass.py:130-144 + eval branch :169-174 on the reference's own modules."""
    cost0 = m.dres0(cost)
    cost0 = m.dres1(cost0) + cost0
    out1, pre1, post1 = m.dres2(cost0, None, None)
    out1 = out1 + cost0
    out2, pre2, post2 = m.dres3(out1, pre1, post1)
    out2 = out2 + cost0
    out3, pre3, post3 = m.dres4(out2, pre1, post2)
    out3 = out3 + cost0
    cost1 = m.classif1(out1)
    cost2 = m.classif2(out2) + cost1
    cost3 = m.classif3(out3) + cost2
    logits = cost3
    c = F.interpolate(cost3, [m.maxdisp - m.mindisp, H, W], mode='trilinear', align_corners=True)
    c = torch.squeeze(c, 1)
    p = F.softmax(c, dim=1)
    return ref_sub.disparityregression(p, m.maxdisp, m.mindisp), logits, cost0


def build_reference(case):
    C = case['C']
    m = PSMNet(case['maxdisp'], case['mindisp'])
    if C != 32:
        m.dres0[0] = ref_sub.convbn_3d(2 * C, 32, 3, 1, 1)  # SURVEY.md section 8c
    m.feature_extraction = nn.Identity()
    sd = recipe.make_state_dict(recipe.stack3d_shapes(C), case['seed'])
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    return m, sd


def calibrate(m, case):
    for mod in m.modules():
        if isinstance(mod, nn.BatchNorm3d):
            mod.momentum = None  # cumulative average -> exact batch statistics
    m.train()
    with torch.no_grad():
        for j in range(2):
            L, R = recipe.make_features(case['B'], case['C'], case['Hf'], case['Wf'], case['seed'] + 100 + j)
            m((L, R))
    m.eval()


def gen_case(name, case):
    torch.manual_seed(0)
    torch.set_num_threads(8)
    m, sd0 = build_reference(case)
    calibrate(m, case)
    L, R = recipe.make_features(case['B'], case['C'], case['Hf'], case['Wf'], case['seed'])
    captured = {}
    hook = m.dres0.register_forward_pre_hook(lambda mod, inp: captured.__setitem__('cost', inp[0].clone()))
    with torch.no_grad():
        pred_genuine = m((L, R))  # reference forward verbatim, H,W = Hf,Wf
    hook.remove()
    cost = captured['cost']
    Hf, Wf = case['Hf'], case['Wf']
    with torch.no_grad():
        pred_g2, logits, cost0 = ref_tail(m, cost, Hf, Wf)
        assert torch.equal(pred_g2, pred_genuine)
        pred_up, _, _ = ref_tail(m, cost, 4 * Hf, 4 * Wf)
        m64 = m.double()
        p64_g, logits64, _ = ref_tail(m64, cost.double(), Hf, Wf)
        p64_up, _, _ = ref_tail(m64, cost.double(), 4 * Hf, 4 * Wf)
    m.float()
    out = dict(
        cost_crc=recipe.checksum(cost), left_crc=recipe.checksum(L), right_crc=recipe.checksum(R),
        pred_genuine=pred_genuine.numpy(), pred_up=pred_up.numpy(), logits=logits.numpy(),
        pred_genuine_f64=p64_g.numpy(), pred_up_f64=p64_up.numpy(), logits_f64=logits64.numpy(),
    )
    if name in ('full', 'live'):  # keep the fixture small: disparity maps only (+ the float64 arbiter's)
        for k in ('logits', 'logits_f64', 'pred_genuine_f64'):
            out.pop(k)
        out['pred_up_f64'] = out['pred_up_f64'].astype(np.float32)
    if name.startswith('tiny'):
        out['cost0'] = cost0.numpy()
    if name == 'tiny_pos':
        out['cost'] = cost.numpy()
    sd = m.state_dict()
    for k, v in sd.items():
        if k.endswith('running_mean') or k.endswith('running_var'):
            out['bn/' + k] = v.numpy()
    # weights checksum over the recipe tensors (regenerated on the GPU box)
    wsum = 0
    for k in sorted(sd0):
        wsum = (wsum * 31 + int(recipe.checksum(sd0[k])[0])) & 0x7FFFFFFFFFFF
    out['weights_crc'] = np.array([wsum], dtype=np.int64)
    e32 = float(np.abs(out['pred_up'] - out['pred_up_f64']).max())
    print(f'{name}: logits std {float(logits.std()):.3f}  ref fp32-vs-fp64 max|d| {e32:.3e}  '
          f'disp range [{float(pred_up.min()):.2f},{float(pred_up.max()):.2f}]')
    out['ref_f32_vs_f64_maxabs'] = np.array([e32])
    np.savez_compressed(os.path.join(HERE, f'idisp_{name}.npz'), **out)


def _weights_crc(sd0):
    wsum = 0
    for k in sorted(sd0):
        wsum = (wsum * 31 + int(recipe.checksum(sd0[k])[0])) & 0x7FFFFFFFFFFF
    return np.array([wsum], dtype=np.int64)


def gen_psm(name, case):
    """The live drop-in call (disprcnn3d.py:266-284 -> stackhourglass.py:106-174): image crop pairs [R,3,224,224] through the
    UNMODIFIED reference PSMNet.forward -- real feature_extraction (submodule.py:60-139) + cost volume + 3-D stack + regression.
    Also stores the reference's own per-view features (forward hook on feature_extraction) for the extractor's parity test."""
    torch.manual_seed(0)
    torch.set_num_threads(8)
    m = PSMNet(case['maxdisp'], case['mindisp'])
    shapes = dict(recipe.stack3d_shapes(32))
    shapes.update(recipe.feature2d_shapes())
    sd0 = recipe.make_state_dict(shapes, case['seed'])
    missing, unexpected = m.load_state_dict(sd0, strict=True)
    for mod in m.modules():
        if isinstance(mod, (nn.BatchNorm2d, nn.BatchNorm3d)):
            mod.momentum = None
    m.train()
    with torch.no_grad():
        for j in range(2):
            L, R = recipe.make_stereo_crops(case['R'], case['size'], case['seed'] + 100 + j)
            m((L, R))
    m.eval()
    L, R = recipe.make_stereo_crops(case['R'], case['size'], case['seed'])
    feas = []
    hook = m.feature_extraction.register_forward_hook(lambda mod, inp, out: feas.append(out.clone()))
    with torch.no_grad():
        pred = m({'left': L, 'right': R})      # dict form, as DispRCNN3D calls it (disprcnn3d.py:273)
        pred_seq = m((L, R))                   # 2-sequence form (stackhourglass.py:110-111)
    hook.remove()
    assert torch.equal(pred, pred_seq) and len(feas) == 4
    with torch.no_grad():
        # float64 arbiter: the reference forward allocates its cost volume as a FloatTensor (stackhourglass.py:117), so the
        # double twin runs the same steps by hand: extractor -> cost volume (oracle restatement of :115-128) -> :130-174
        import idispnet_oracle as O
        m64 = m.double()
        f64 = [m64.feature_extraction(L.double()), m64.feature_extraction(R.double())]
        cost64 = O.cost_volume(f64[0], f64[1], case['mindisp'], case['maxdisp'])
        pred64, _, _ = ref_tail(m64, cost64, case['size'], case['size'])
    m.float()
    with torch.no_grad():  # the same hand-run chain in float32 reproduces the genuine forward bit for bit
        p32, _, _ = ref_tail(m, O.cost_volume(feas[0], feas[1], case['mindisp'], case['maxdisp']), case['size'], case['size'])
        assert torch.equal(p32, pred)
    out = dict(pred=pred.numpy(), pred_f64=pred64.numpy().astype(np.float32), fea_left=feas[0].numpy(), fea_right=feas[1].numpy(),
               fea_left_f64=f64[0].numpy().astype(np.float32),
               left_crc=recipe.checksum(L), right_crc=recipe.checksum(R), weights_crc=_weights_crc(sd0))
    for k, v in m.state_dict().items():
        if k.endswith('running_mean') or k.endswith('running_var'):
            out['bn/' + k] = v.numpy()
    e32 = float(np.abs(out['pred'] - pred64.numpy()).max())
    ef = float(np.abs(out['fea_left'] - f64[0].numpy()).max())
    out['ref_f32_vs_f64_maxabs'] = np.array([e32])
    print(f'{name}: disp range [{float(pred.min()):.2f},{float(pred.max()):.2f}] std {float(pred.std()):.2f}; ref fp32-vs-fp64 max|d| {e32:.3e}; '
          f'features |max| {float(feas[0].abs().max()):.2f}, fp32-vs-fp64 {ef:.3e}')
    np.savez_compressed(os.path.join(HERE, f'{name}.npz'), **out)


def gen_raw(name, case):
    """Default-initialised weights (stackhourglass.py:90-104; SURVEY.md section 8c): no calibration, nothing damped -- logits of std
    ~17, where the reference's own fp32 forward is already ~3e-3 px from its float64 twin."""
    torch.manual_seed(0)
    torch.set_num_threads(8)
    m = PSMNet(case['maxdisp'], case['mindisp'])
    m.feature_extraction = nn.Identity()
    sd0 = recipe.make_state_dict(recipe.stack3d_shapes(case['C']), case['seed'], raw=True)
    missing, unexpected = m.load_state_dict(sd0, strict=False)
    assert not missing and not unexpected, (missing, unexpected)
    m.eval()
    L, R = recipe.make_features(case['B'], case['C'], case['Hf'], case['Wf'], case['seed'])
    captured = {}
    hook = m.dres0.register_forward_pre_hook(lambda mod, inp: captured.__setitem__('cost', inp[0].clone()))
    with torch.no_grad():
        pred_genuine = m((L, R))
    hook.remove()
    cost = captured['cost']
    Hf, Wf = case['Hf'], case['Wf']
    with torch.no_grad():
        pred_up, logits, _ = ref_tail(m, cost, 4 * Hf, 4 * Wf)
        m64 = m.double()
        p64_up, logits64, _ = ref_tail(m64, cost.double(), 4 * Hf, 4 * Wf)
        p64_g, _, _ = ref_tail(m64, cost.double(), Hf, Wf)
    m.float()
    e32 = float(np.abs(pred_up.numpy() - p64_up.numpy()).max())
    out = dict(pred_up=pred_up.numpy(), pred_genuine=pred_genuine.numpy(), pred_up_f64=p64_up.numpy().astype(np.float32),
               pred_genuine_f64=p64_g.numpy().astype(np.float32),
               left_crc=recipe.checksum(L), right_crc=recipe.checksum(R), weights_crc=_weights_crc(sd0),
               ref_f32_vs_f64_maxabs=np.array([e32]), logits_std=np.array([float(logits.std())]))
    print(f'{name}: logits std {float(logits.std()):.3f}  ref fp32-vs-fp64 max|d| {e32:.3e}  disp range [{float(pred_up.min()):.2f},{float(pred_up.max()):.2f}]')
    np.savez_compressed(os.path.join(HERE, f'{name}.npz'), **out)


def gen_paste(name, case):
    """SURVEY.md 8(f) row 3: the per-ROI disparity hand-off, produced by EXECUTING the reference's own ``DisparityMap.resize`` /
    ``.crop`` (disprcnn/structures/disparity.py:39-78; importable once disprcnn_b200.install() has put the ``disprcnn._C`` shim in
    place -- ``disprcnn.layers`` is what it imports) inside the two loops that call it, restated here line by line:
    ``DispRCNN3D.roi_disp_postprocess`` (disprcnn3d.py:161-190) and the depth part of ``PointRCNN.process_input``
    (point_rcnn.py:113-136)."""
    import warnings
    import disprcnn_b200
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        disprcnn_b200.install(inference_only=True)
    from disprcnn.structures.disparity import DisparityMap   # the reference class
    from disprcnn.utils.stereo_utils import expand_box_to_integer
    disp, lbs, rbs, masks, fub = recipe.make_paste_inputs(case)
    H, W = case['H'], case['W']
    maps, depths, r = [], [], 0
    for lb_img, rb_img in zip(lbs, rbs):
        roi_disps_per_img = []
        for leftbox, rightbox in zip(lb_img, rb_img):
            x1, y1, x2, y2 = expand_box_to_integer(leftbox)
            x1p, _, x2p, _ = expand_box_to_integer(rightbox)
            roi_disp = DisparityMap(disp[r]).resize((max(x2 - x1, x2p - x1p), y2 - y1)).crop((0, 0, x2 - x1, y2 - y1))     # disprcnn3d.py:173-175
            disparity_map_per_roi = torch.zeros((H, W))
            disparity_map_per_roi[int(y1):int(y1) + roi_disp.height, int(x1):int(x1) + roi_disp.width] = roi_disp.data + (x1 - x1p)
            disparity_map_per_roi = disparity_map_per_roi.clone().clamp(min=0)
            disparity_map_per_roi = disparity_map_per_roi * masks[r].float()
            roi_disps_per_img.append(disparity_map_per_roi)
            # point_rcnn.py:124-134
            depth_map_per_roi = torch.zeros((H, W))
            disp_roi = DisparityMap(disp[r]).resize((max(x2 - x1, x2p - x1p), y2 - y1)).crop((0, 0, x2 - x1, y2 - y1)).data
            disp_roi = disp_roi + x1 - x1p
            depth_roi = float(fub[r]) / (disp_roi + 1e-6)
            depth_map_per_roi[y1:y2, x1:x2] = depth_roi
            depths.append(depth_map_per_roi)
            r += 1
        maps.append(torch.stack(roi_disps_per_img).max(dim=0)[0] if roi_disps_per_img else torch.zeros((H, W)))
    out = dict(disparity_maps=torch.stack(maps).numpy(), depth_maps=torch.stack(depths).numpy(), disp_crc=recipe.checksum(disp),
               mask_crc=recipe.checksum(masks))
    print(f'{name}: {len(depths)} ROIs on {len(maps)} images {H}x{W}; disparity map max {float(torch.stack(maps).max()):.2f}')
    np.savez_compressed(os.path.join(HERE, f'{name}.npz'), **out)


def gen_roi():
    import build_ref
    ref = build_ref.build()
    for name, rc in recipe.ROI_CASES.items():
        g = recipe._gen(rc['seed'], 'roi_input')
        inp = torch.randn(rc['N'], rc['C'], rc['H'], rc['W'], generator=g)
        rois = torch.tensor(rc['rois'], dtype=torch.float32)
        out = ref.roi_align_forward(inp, rois, rc['scale'], rc['ph'], rc['pw'], rc['sr'])
        np.savez_compressed(os.path.join(HERE, f'roialign_{name}.npz'), out=out.numpy(),
                            input_crc=recipe.checksum(inp))
        print(f'roialign {name}: out {tuple(out.shape)}')
    inp, rois = recipe.make_random_roi_inputs()
    out = {'input_crc': recipe.checksum(inp), 'rois_crc': recipe.checksum(rois)}
    for i, (ph, pw, sc, sr) in enumerate(recipe.ROI_RANDOM_CONFIGS):
        out[f'out{i}'] = ref.roi_align_forward(inp, rois, sc, ph, pw, sr).numpy()
    np.savez_compressed(os.path.join(HERE, 'roialign_random.npz'), **out)
    print(f'roialign random: {len(recipe.ROI_RANDOM_CONFIGS)} pooling configs')


if __name__ == '__main__':
    which = sys.argv[1:] or list(recipe.CASES) + list(recipe.PSM_CASES) + list(recipe.RAW_CASES) + list(recipe.PASTE_CASES) + ['roi']
    for name in which:
        if name == 'roi':
            gen_roi()
        elif name in recipe.PSM_CASES:
            gen_psm(name, recipe.PSM_CASES[name])
        elif name in recipe.RAW_CASES:
            gen_raw(name, recipe.RAW_CASES[name])
        elif name in recipe.PASTE_CASES:
            gen_paste(name, recipe.PASTE_CASES[name])
        else:
            gen_case(name, recipe.CASES[name])
