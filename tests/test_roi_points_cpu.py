"""CPU: the per-ROI point-cloud hand-off without a GPU -- the host sampler against numpy, the oracle against the fixture made by
executing the reference's PointRCNN.process_input_eval, and the argument checks of the three C entry points."""
import ctypes
import os

import numpy as np
import pytest
import torch

import points_oracle as PO
import points_recipe as PR

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _choice(lib, n, P):
    out = np.full(P, -7, np.int32)
    assert lib.idisp_roi_points_choice(n, P, out.ctypes.data_as(ctypes.c_void_p)) == 0
    return out


def test_choice_matches_numpy(built_lib):
    """idisp_roi_points_choice == back_project's np.random.seed(0) / choice / seed(0) / shuffle (point_rcnn.py:53-74), bit for bit."""
    for n in list(range(1, 3001)) + [4095, 4096, 4097, 10 ** 5, 375 * 1242]:
        assert np.array_equal(_choice(built_lib, n, 768), PO.choice(n, 768)), n
    for P in (1, 16, 1024):
        for n in (1, 2, P - 1, P, P + 1, 3 * P + 5, 5000):
            if n >= 1:
                assert np.array_equal(_choice(built_lib, n, P), PO.choice(n, P)), (n, P)


def load_points_case(name):
    case = PR.POINTS_CASES[name]
    g = np.load(os.path.join(GOLDEN, f'{name}.npz'))
    disp, probs, lb, rb, counts, P2s, P3s = PR.make_points_inputs(case, int(g['seed'][0]))
    assert np.array_equal(PR.checksums(disp, probs, lb, rb), g['input_crc']), 'regenerated inputs differ from the golden ones'
    from disprcnn_b200.layers.roi_points import calib_row
    calibs = [calib_row(a, b) for a, b in zip(P2s, P3s)]
    sizes = [img['size'] for img in case['images']]
    return case, g, (disp, probs, lb, rb, counts, calibs, sizes)


def test_oracle_matches_reference_fixture():
    case, g, (disp, probs, lb, rb, counts, calibs, sizes) = load_points_case('points_kitti')
    pts, mean, rot, pix, n = PO.roi_points(disp, probs, lb, rb, counts, calibs, sizes, case['npoints'])
    assert np.array_equal(n.numpy(), g['counts']) and np.array_equal(pix.numpy(), g['pixels'])
    assert np.abs(pts.numpy() - g['pts']).max() <= 1e-4 * max(1.0, float(np.abs(g['pts']).max()))
    assert np.abs(mean.numpy() - g['pts_mean']).max() <= 1e-4 * max(1.0, float(np.abs(g['pts_mean']).max()))
    assert np.array_equal(rot.numpy(), g['rot_angle'])
    # the Masker's masks, exactly
    r = 0
    for i, (W, H) in enumerate(sizes):
        want = np.unpackbits(g[f'masks{i}'], axis=1)[:, :H * W].reshape(-1, H, W)
        for k in range(counts[i]):
            assert np.array_equal(PO.paste_mask(probs[r, 0], lb[r], H, W).numpy(), want[k]), r
            r += 1
    # the fixture covers n > P, n < P and n == P
    assert (g['counts'] > 768).any() and (g['counts'] < 768).any() and (g['counts'] == 768).any()


def test_argument_validation_without_gpu(built_lib):
    lib = built_lib
    from disprcnn_b200 import _lib
    buf = ctypes.c_void_p(1)   # never dereferenced: every call below fails its checks before touching memory
    out = np.zeros(4, np.int32)
    op = out.ctypes.data_as(ctypes.c_void_p)
    # sampler
    assert lib.idisp_roi_points_choice(0, 768, op) == 1 and 'positive' in _lib.last_error()
    assert lib.idisp_roi_points_choice(5, 0, op) == 1
    assert lib.idisp_roi_points_choice(5, -3, op) == 1
    assert lib.idisp_roi_points_choice(5, 4, None) == 1 and 'NULL' in _lib.last_error()

    def count(R=1, S=224, M=28, n_images=1, thr=0.5, pad=1, ptr=buf, cnt=buf):
        return lib.idisp_roi_points_count(ptr, R, S, ptr, M, ptr, ptr, ptr, ptr, ptr, n_images, thr, pad, cnt, None)

    def gather(R=1, S=224, M=28, n_images=1, thr=0.5, pad=1, P=768, ptr=buf, pts=buf, max_depth=160.0):
        return lib.idisp_roi_points_gather(ptr, R, S, ptr, M, ptr, ptr, ptr, ptr, ptr, n_images, thr, pad, ptr, ptr, P, max_depth, pts,
                                           ptr, ptr, None, None)
    for fn in (count, gather):
        assert fn(R=0) == 0                                            # R == 0: no-op, nothing launched
        assert fn(ptr=None) == 1 and 'NULL' in _lib.last_error()
        assert fn(R=-1) == 1 and 'bad shape' in _lib.last_error()
        assert fn(S=0) == 1 and fn(M=0) == 1
        assert fn(pad=0) == 1 and 'padding' in _lib.last_error()
        assert fn(M=127) == 1                                          # padded mask side over the limit
        assert fn(thr=-0.5) == 1 and 'threshold' in _lib.last_error()
        assert fn(n_images=0) == 1
    assert count(cnt=None) == 1
    assert gather(pts=None) == 1
    assert gather(P=0) == 1 and 'npoints' in _lib.last_error()
    assert gather(P=-5) == 1 and gather(P=16385) == 1
    assert gather(R=0, P=0) == 1                                       # npoints is checked even for R == 0
    assert gather(max_depth=float('nan')) == 1


def test_python_layer_refuses_cpu_tensors(built_lib):
    from disprcnn_b200.layers import roi_points
    d, m, b = torch.zeros(1, 8, 8), torch.zeros(1, 1, 4, 4), torch.tensor([[0., 0., 4., 4.]])
    with pytest.raises(RuntimeError, match='no CPU path'):
        roi_points(d, m, b, b, [1], [[700., 700., 600., 170., 0., 0., 380.]], [(64, 32)])
