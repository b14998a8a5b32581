"""Timing of the per-ROI point-cloud hand-off (disprcnn_b200.layers.roi_points, csrc/roi_points.cu) on one GPU.

R = 1 / 4 / 8 / 15 ROIs over 375 x 1242 images (at most five ROIs per image), S = 224 disparity maps, M = 28 masks, P = 768.
Per R: the count kernel and the H2D + gather (CUDA events), the D2H of the counts + host sampler (host clock, after the count
kernel has finished), and the whole ``roi_points`` call (host clock ending in a synchronise) -- every figure the median of --reps
runs after --warmup.  The reference-shaped baseline is the test oracle (tests/golden/points_oracle.py: image-sized maps per ROI,
depthmap_to_rect over the image, numpy sampling) run eagerly on the same GPU, after asserting that both agree.

usage: python tools/bench_points.py --out profiles/r03_points_bench.json [--reps 50] [--warmup 5]
"""
import argparse
import json
import os
import subprocess
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tests', 'golden'), os.path.join(ROOT, 'oracle')):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import points_oracle as PO  # noqa: E402
import points_recipe as PR  # noqa: E402
from disprcnn_b200 import _lib  # noqa: E402
from disprcnn_b200.layers.roi_points import calib_row, roi_points  # noqa: E402


def power_limit():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as e:   # the figure is reported, never required
        return f'unavailable ({e})'


def staged(lib, d, p, lb, rb, idx, wh, cal, N, P):
    """roi_points step by step with a timer around each step; returns (count_ms, d2h_sampler_ms, h2d_gather_ms)."""
    R, S, M = d.shape[0], d.shape[-1], p.shape[-1]
    args = (_lib.ptr(d), R, S, _lib.ptr(p), M, _lib.ptr(lb), _lib.ptr(rb), _lib.ptr(idx), _lib.ptr(wh), _lib.ptr(cal), N, 0.5, 1)
    count = torch.empty((R,), dtype=torch.int32, device='cuda')
    pts = torch.empty((R, P, 3), device='cuda')
    mean = torch.empty((R, 3), device='cuda')
    rot = torch.empty((R,), dtype=torch.float64, device='cuda')
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e[0].record()
    _lib.check(lib.idisp_roi_points_count(*args, _lib.ptr(count), _lib.stream_ptr()))
    e[1].record()
    e[1].synchronize()
    t0 = time.perf_counter()
    n = count.cpu().tolist()
    ranks = torch.empty((R, P), dtype=torch.int32, pin_memory=True)
    for r, c in enumerate(n):
        _lib.check(lib.idisp_roi_points_choice(c, P, _lib.ptr(ranks[r])))
    t1 = time.perf_counter()
    e[2].record()
    ranks = ranks.to('cuda', non_blocking=True)
    _lib.check(lib.idisp_roi_points_gather(*args, _lib.ptr(count), _lib.ptr(ranks), P, 160.0, _lib.ptr(pts), _lib.ptr(mean), _lib.ptr(rot),
                                           None, _lib.stream_ptr()))
    e[3].record()
    e[3].synchronize()
    return e[0].elapsed_time(e[1]), (t1 - t0) * 1e3, e[2].elapsed_time(e[3])


def host_ms(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--reps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--oracle-reps', type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_points.py measures on a CUDA device; there is no CPU figure'
    lib = _lib.load()
    res = dict(gpu=torch.cuda.get_device_name(0), power_limit=power_limit(), torch=torch.__version__, shape=dict(H=375, W=1242, S=224, M=28,
               npoints=768), reps=a.reps, warmup=a.warmup, oracle_reps=a.oracle_reps, runs=[])
    P = 768
    for R in (1, 4, 8, 15):
        per = [min(5, R - 5 * i) for i in range((R + 4) // 5)]
        disp, probs, lb, rb, counts, P2s, P3s, sizes = PR.make_kitti_batch(per, 90 + R)
        calibs = [calib_row(x, y) for x, y in zip(P2s, P3s)]
        d, p, l, r = disp.cuda(), probs.cuda(), lb.cuda(), rb.cuda()
        p3 = p.reshape(R, 28, 28).contiguous()
        idx = torch.repeat_interleave(torch.arange(len(per), dtype=torch.int32), torch.tensor(per)).cuda()
        wh = torch.tensor(sizes, dtype=torch.int32).cuda()
        cal = torch.tensor(np.asarray(calibs, np.float64)).cuda()
        call = lambda: roi_points(d, p, l, r, counts, calibs, sizes, P, return_pixels=True)  # noqa: E731
        got = call()
        ora = PO.roi_points(d, p, l, r, counts, calibs, sizes, P)
        assert torch.equal(got[3].long(), ora[3]), f'R={R}: chosen pixels differ from the oracle'
        err = float((got[0] - ora[0]).abs().max() / max(1.0, float(ora[0].abs().max())))
        assert err <= 1e-4, f'R={R}: pts differ from the oracle by {err}'
        for _ in range(a.warmup):
            call()
            staged(lib, d, p3, l, r, idx, wh, cal, len(per), P)
        whole = [host_ms(call) for _ in range(a.reps)]
        st = [staged(lib, d, p3, l, r, idx, wh, cal, len(per), P) for _ in range(a.reps)]
        host_ms(lambda: PO.roi_points(d, p, l, r, counts, calibs, sizes, P))   # warm-up
        oracle = [host_ms(lambda: PO.roi_points(d, p, l, r, counts, calibs, sizes, P)) for _ in range(a.oracle_reps)]
        med = statistics.median
        run = dict(R=R, images=len(per), points=ora[4].tolist(), call_ms=med(whole), call_ms_min=min(whole),
                   count_kernel_ms=med([s[0] for s in st]), d2h_sampler_ms=med([s[1] for s in st]), h2d_gather_ms=med([s[2] for s in st]),
                   oracle_eager_ms=med(oracle), speedup_vs_oracle=med(oracle) / med(whole), pts_rel_err_vs_oracle=err)
        res['runs'].append(run)
        print(json.dumps(run))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=res['gpu'], power_limit=res['power_limit'])))


if __name__ == '__main__':
    main()
