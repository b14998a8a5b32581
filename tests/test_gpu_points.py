"""GPU: csrc/roi_points.cu (per-ROI point clouds for PointRCNN) against the fixture made by executing the reference's
PointRCNN.process_input_eval, against the oracle on a KITTI-size batch, and its error paths."""
import types

import numpy as np
import pytest
import torch

import points_oracle as PO
import points_recipe as PR
from test_roi_points_cpu import load_points_case

pytestmark = pytest.mark.gpu


def _rel(got, want):
    return float(np.abs(got - want).max() / max(1.0, float(np.abs(want).max())))


def _batch(R_per_image, seed):
    from disprcnn_b200.layers.roi_points import calib_row
    disp, probs, lb, rb, counts, P2s, P3s, sizes = PR.make_kitti_batch(R_per_image, seed)
    return disp, probs, lb, rb, counts, [calib_row(a, b) for a, b in zip(P2s, P3s)], sizes


def _cuda(disp, probs, lb, rb):
    return disp.cuda(), probs.cuda(), lb.cuda(), rb.cuda()


def test_points_against_reference_fixture():
    from disprcnn_b200.layers import roi_points
    case, g, (disp, probs, lb, rb, counts, calibs, sizes) = load_points_case('points_kitti')
    pts, mean, rot, pix = roi_points(*_cuda(disp, probs, lb, rb), counts, calibs, sizes, case['npoints'], return_pixels=True)
    pts, mean, rot, pix = pts.cpu().numpy(), mean.cpu().numpy(), rot.cpu().numpy(), pix.cpu().numpy()
    e_pts, e_mean = _rel(pts, g['pts']), _rel(mean, g['pts_mean'])
    e_rot = float((np.abs(rot - g['rot_angle']) / np.maximum(np.abs(g['rot_angle']), 1e-300)).max())
    print(f'\n[points] pixels equal: {np.array_equal(pix, g["pixels"])}; pts max |d| / max(1, |ref|) {e_pts:.3e}; '
          f'pts_mean {e_mean:.3e}; rot_angle max rel {e_rot:.3e}')
    assert np.array_equal(pix, g['pixels'])
    assert e_pts <= 1e-4 and e_mean <= 1e-4 and e_rot <= 1e-12
    assert rot.dtype == np.float64
    # the counts exactly: the count kernel on its own
    n = _count(disp, probs, lb, rb, counts, calibs, sizes)
    assert np.array_equal(n, g['counts']), (n, g['counts'])


def _count(disp, probs, lb, rb, counts, calibs, sizes):
    from disprcnn_b200 import _lib
    R = disp.shape[0]
    d, p, l, r = _cuda(disp, probs.reshape(R, probs.shape[-1], -1).contiguous(), lb, rb)
    idx = torch.repeat_interleave(torch.arange(len(counts), dtype=torch.int32), torch.tensor(counts)).cuda()
    wh = torch.tensor(sizes, dtype=torch.int32).cuda()
    cal = torch.tensor(np.asarray(calibs, np.float64)).cuda()
    out = torch.empty(R, dtype=torch.int32, device='cuda')
    _lib.check(_lib.load().idisp_roi_points_count(_lib.ptr(d), R, d.shape[-1], _lib.ptr(p), p.shape[-1], _lib.ptr(l), _lib.ptr(r),
                                                  _lib.ptr(idx), _lib.ptr(wh), _lib.ptr(cal), len(counts), 0.5, 1, _lib.ptr(out),
                                                  _lib.stream_ptr()))
    return out.cpu().numpy()


def test_points_against_oracle_kitti_batch():
    """R = 15 over three 375 x 1242 images, the middle one without ROIs; plus: bit-identical on a repeat call, and no image-sized
    allocation."""
    from disprcnn_b200.layers import roi_points
    disp, probs, lb, rb, counts, calibs, sizes = _batch([9, 0, 6], 81)
    pts_o, mean_o, rot_o, pix_o, n_o = PO.roi_points(disp, probs, lb, rb, counts, calibs, sizes)
    args = _cuda(disp, probs, lb, rb)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    pts, mean, rot, pix = roi_points(*args, counts, calibs, sizes, return_pixels=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < 375 * 1242 * 4, f'{peak} B allocated: as much as an image-sized f32 map'
    e_pts, e_mean = _rel(pts.cpu().numpy(), pts_o.numpy()), _rel(mean.cpu().numpy(), mean_o.numpy())
    e_rot = float((rot.cpu() - rot_o).abs().max() / rot_o.abs().max())
    print(f'\n[points R=15] n {n_o.tolist()}; pts {e_pts:.3e}, pts_mean {e_mean:.3e}, rot_angle {e_rot:.3e}; peak alloc {peak} B')
    assert np.array_equal(pix.cpu().numpy(), pix_o.numpy())
    assert e_pts <= 1e-4 and e_mean <= 1e-4 and e_rot <= 1e-12
    again = roi_points(*args, counts, calibs, sizes, return_pixels=True)
    for a, b in zip((pts, mean, rot, pix), again):
        assert torch.equal(a, b)


def test_points_empty_and_npoints():
    from disprcnn_b200.layers import roi_points
    disp, probs, lb, rb, counts, calibs, sizes = _batch([0, 0], 82)
    pts, mean, rot = roi_points(*_cuda(disp, probs, lb, rb), counts, calibs, sizes)
    assert pts.shape == (0, 768, 3) and mean.shape == (0, 3) and rot.shape == (0,)
    # another P, against the oracle
    disp, probs, lb, rb, counts, calibs, sizes = _batch([2, 1], 83)
    pts, mean, rot, pix = roi_points(*_cuda(disp, probs, lb, rb), counts, calibs, sizes, npoints=100, return_pixels=True)
    pts_o, mean_o, _, pix_o, _ = PO.roi_points(disp, probs, lb, rb, counts, calibs, sizes, npoints=100)
    assert pts.shape == (3, 100, 3) and np.array_equal(pix.cpu().numpy(), pix_o.numpy())
    assert _rel(pts.cpu().numpy(), pts_o.numpy()) <= 1e-4


def test_points_error_paths():
    from disprcnn_b200.layers import roi_points
    disp, probs, lb, rb, counts, calibs, sizes = _batch([2, 1], 84)

    def run(lb_=lb, disp_=disp):
        return roi_points(*_cuda(disp_, probs, lb_, rb), counts, calibs, sizes)
    bad = lb.clone()
    bad[1] = torch.tensor([1200.0, 10.0, 1250.5, 60.0])            # reaches past the 1242-px image
    with pytest.raises(RuntimeError, match='ROI 1 .*not inside its image'):
        run(lb_=bad)
    bad = lb.clone()
    bad[2] = torch.tensor([300.0, 40.0, 300.0, 90.0])              # zero-width box: no point at all
    with pytest.raises(ValueError, match='ROI 2: mask is nonvalid'):
        run(lb_=bad)
    nan = disp.clone()
    nan[0, 90:130, 90:130] = float('nan')                        # wider than the resize's sampling step
    with pytest.raises(RuntimeError, match='ROI 0 .*not finite'):
        run(disp_=nan)
    run()   # and the good batch still goes through after the failures


def test_process_input_eval_mirror():
    """The reference method's signature on duck-typed BoxList-like inputs gives what roi_points gives."""
    from disprcnn_b200.layers import process_input_eval, roi_points
    disp, probs, lb, rb, counts, calibs, sizes = _batch([3, 0, 2], 85)
    base = PR.POINTS_CASES['points_kitti']['images'][0]

    class Box:
        def __init__(self, bbox, size, fields):
            self.bbox, self.size, self._f = bbox, size, fields

        def get_field(self, k):
            return self._f[k]
    lefts, rights, targets, r0 = [], [], [], 0
    for c, size in zip(counts, sizes):
        sl = slice(r0, r0 + c)
        r0 += c
        lefts.append(Box(lb[sl].cuda(), size, {'disparity': disp[sl].cuda(), 'mask': probs[sl].cuda()}))
        rights.append(Box(rb[sl].cuda(), size, {}))
        calib = types.SimpleNamespace(calib=types.SimpleNamespace(P2=np.asarray(base['P2']), P3=np.asarray(base['P3'])))
        targets.append(Box(None, size, {'calib': calib}))
    got = process_input_eval(lefts, rights, targets, threshold=0.5)
    want = roi_points(*_cuda(disp, probs, lb, rb), counts, calibs, sizes)
    for a, b in zip(got, want):
        assert torch.equal(a, b)
