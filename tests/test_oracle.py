"""CPU: the oracle restatement against the golden vectors produced by executing the reference."""
import ctypes
import os

import numpy as np
import pytest
import torch

import idispnet_oracle as O
import recipe
from helpers import GOLDEN, load_case, load_psm_case, load_raw_case

ORACLE_DIR = os.path.dirname(os.path.abspath(O.__file__))


@pytest.mark.parametrize('name', ['tiny', 'tiny_pos', 'c1', 'live'])
def test_cost_volume_matches_reference(name):
    case, g, sd, L, R = load_case(name)
    cost = O.cost_volume(L, R, case['mindisp'], case['maxdisp'])
    assert int(recipe.checksum(cost)[0]) == int(g['cost_crc'][0])  # bit-exact copy semantics
    if 'cost' in g.files:
        assert np.array_equal(cost.numpy(), g['cost'])


@pytest.mark.parametrize('name', ['tiny', 'tiny_pos', 'c1', 'live'])
def test_stack_and_regression_match_reference(name):
    case, g, sd, L, R = load_case(name)
    torch.set_num_threads(8)
    with torch.no_grad():
        cost = O.cost_volume(L, R, case['mindisp'], case['maxdisp'])
        logits, inter = O.stack3d(cost, sd, return_intermediates=True)
        up = O.upsample_softargmin(logits, case['mindisp'], case['maxdisp'], 4 * case['Hf'], 4 * case['Wf'])
        gen = O.upsample_softargmin(logits, case['mindisp'], case['maxdisp'], case['Hf'], case['Wf'])
    # same torch CPU ops as the reference modules -> agreement far below the 1e-3 parity tolerance
    if 'logits' in g.files:   # (the larger fixtures keep only the disparity maps)
        assert np.abs(logits.numpy() - g['logits']).max() < 2e-5
    assert np.abs(up.numpy() - g['pred_up']).max() < 5e-5
    assert np.abs(gen.numpy() - g['pred_genuine']).max() < 5e-5
    if 'cost0' in g.files:
        assert np.abs(inter['cost0'].numpy() - g['cost0']).max() < 2e-5
    # and the reference itself sits this far from its float64 twin (context for the tolerance)
    assert float(g['ref_f32_vs_f64_maxabs'][0]) < 1e-3


def test_disparityregression_and_full_entry():
    case, g, sd, L, R = load_case('tiny')
    with torch.no_grad():
        out = O.idispnet_from_features(L, R, sd, case['mindisp'], case['maxdisp'])
    assert np.abs(out.numpy() - g['pred_up']).max() < 5e-5
    p = torch.softmax(torch.randn(2, 32, 3, 5), 1)
    ref = sum(p[:, d] * float(-16 + d) for d in range(32))
    assert torch.allclose(O.disparityregression(p, 16, -16), ref, atol=1e-5)


def test_feature_extraction_and_whole_psmnet_match_reference():
    """The live drop-in call: image crops through the extractor restatement (submodule.py:60-139) and the rest of the path,
    against the features and the disparity the UNMODIFIED reference PSMNet.forward produced (tests/golden/psm_live.npz)."""
    case, g, sd, L, R = load_psm_case('psm_live')
    torch.set_num_threads(8)
    with torch.no_grad():
        fl = O.feature_extraction(L, sd)
        fr = O.feature_extraction(R, sd)
        pred = O.idispnet_from_features(fl, fr, sd, case['mindisp'], case['maxdisp'], case['size'], case['size'])
    assert np.abs(fl.numpy() - g['fea_left']).max() < 2e-5 and np.abs(fr.numpy() - g['fea_right']).max() < 2e-5
    assert np.abs(pred.numpy() - g['pred']).max() < 5e-5
    assert float(g['ref_f32_vs_f64_maxabs'][0]) < 1e-3


@pytest.mark.parametrize('name', ['raw_tiny', 'raw_live'])
def test_default_initialised_stack_matches_reference(name):
    """SURVEY.md 8(c): the raw default-init fixture next to the trained-like ones (logit std ~15: the reference's own fp32
    forward is up to 2.5e-3 px from its float64 twin there -- stored in the fixture)."""
    case, g, sd, L, R = load_raw_case(name)
    torch.set_num_threads(8)
    with torch.no_grad():
        up = O.idispnet_from_features(L, R, sd, case['mindisp'], case['maxdisp'])
    assert np.abs(up.numpy() - g['pred_up']).max() < 2e-4
    assert float(g['logits_std'][0]) > 10


def _roi_inputs(rc):
    g = recipe._gen(rc['seed'], 'roi_input')
    inp = torch.randn(rc['N'], rc['C'], rc['H'], rc['W'], generator=g)
    return inp, np.asarray(rc['rois'], dtype=np.float32)


@pytest.mark.parametrize('name', list(recipe.ROI_CASES))
def test_roi_align_numpy_oracle_bit_exact(name):
    rc = recipe.ROI_CASES[name]
    gold = np.load(os.path.join(GOLDEN, f'roialign_{name}.npz'))
    inp, rois = _roi_inputs(rc)
    assert int(recipe.checksum(inp)[0]) == int(gold['input_crc'][0])
    out = O.roi_align_forward(inp.numpy(), rois, rc['scale'], rc['ph'], rc['pw'], rc['sr'])
    assert np.array_equal(out, gold['out'])


@pytest.mark.parametrize('name', list(recipe.ROI_CASES))
def test_roi_align_c_oracle_bit_exact(name):
    so = os.path.join(ORACLE_DIR, '_build', 'liboracle.so')
    if not os.path.exists(so):
        import subprocess
        subprocess.check_call(['make', '-C', ORACLE_DIR, '-s'])
    lib = ctypes.CDLL(so)
    rc = recipe.ROI_CASES[name]
    gold = np.load(os.path.join(GOLDEN, f'roialign_{name}.npz'))
    inp, rois = _roi_inputs(rc)
    x = np.ascontiguousarray(inp.numpy())
    out = np.zeros_like(gold['out'])
    fp = ctypes.POINTER(ctypes.c_float)
    lib.oracle_roi_align_forward(x.ctypes.data_as(fp), rc['N'], rc['C'], rc['H'], rc['W'], rois.ctypes.data_as(fp),
                                 len(rois), ctypes.c_float(rc['scale']), rc['ph'], rc['pw'], rc['sr'],
                                 out.ctypes.data_as(fp))
    assert np.array_equal(out, gold['out'])


def test_roi_align_against_compiled_reference_if_present():
    """The reference's own CPU kernel on random boxes: its stored outputs (tests/golden/roialign_random.npz), and the kernel
    itself where oracle/_ref holds a build of it (python oracle/build_ref.py)."""
    import build_ref
    gold = np.load(os.path.join(GOLDEN, 'roialign_random.npz'))
    inp, rois = recipe.make_random_roi_inputs()
    assert int(recipe.checksum(inp)[0]) == int(gold['input_crc'][0]) and int(recipe.checksum(rois)[0]) == int(gold['rois_crc'][0])
    ref = build_ref.load_prebuilt()
    for i, (ph, pw, sc, sr) in enumerate(recipe.ROI_RANDOM_CONFIGS):
        b = O.roi_align_forward(inp.numpy(), rois.numpy(), sc, ph, pw, sr)
        assert np.array_equal(gold[f'out{i}'], b)
        if ref is not None:
            assert np.array_equal(ref.roi_align_forward(inp, rois, sc, ph, pw, sr).numpy(), b)


def test_crop_normalise_and_box_alignment():
    im = recipe.make_images(1, 40, 64, 3).numpy()
    rl, rr = O.align_stereo_boxes([[(10.2, 5.7, 30.1, 25.3)]], [[(4.9, 5.0, 22.0, 26.0)]], 64, 40)
    assert rl == [[0, 10, 5, 31, 26]] and rr == [[0, 4, 5, 25, 26]]
    out = O.crop_and_transform_roi_img(im, np.asarray(rl, np.float32), 16)
    raw = O.roi_align_forward(im, np.asarray(rl, np.float32), 1.0, 16, 16, 0)
    m = np.asarray(O.IMAGENET_MEAN, np.float32)[None, :, None, None]
    s = np.asarray(O.IMAGENET_STD, np.float32)[None, :, None, None]
    assert np.array_equal(out, (raw - m) / s)


def test_roi_disparity_handoff_matches_reference():
    """SURVEY.md 8(f) row 3: resize / crop / shift / clamp / mask / max of the per-ROI disparity maps and the depth maps, against the
    fixture made by executing the reference's DisparityMap inside its two call-site loops (tests/golden/paste_small.npz)."""
    case = recipe.PASTE_CASES['paste_small']
    g = np.load(os.path.join(GOLDEN, 'paste_small.npz'))
    disp, lbs, rbs, masks, fub = recipe.make_paste_inputs(case)
    assert int(recipe.checksum(disp)[0]) == int(g['disp_crc'][0]) and int(recipe.checksum(masks)[0]) == int(g['mask_crc'][0])
    maps = O.roi_disp_postprocess(disp, lbs, rbs, masks, case['H'], case['W'])
    flat_l, flat_r = [b for im in lbs for b in im], [b for im in rbs for b in im]
    depth = O.roi_depth_maps(disp, flat_l, flat_r, fub, case['H'], case['W'])
    assert np.array_equal(maps.numpy(), g['disparity_maps'])     # same torch CPU ops in the same order
    assert np.array_equal(depth.numpy(), g['depth_maps'])
    assert maps.shape == (3, case['H'], case['W']) and float(maps[2].abs().max()) == 0.0   # image without ROIs -> zero map
