"""ctypes binding of libidisp.so (the C-ABI declared in include/idisp.h) + its in-tree build.

The library is the product; this module only loads it, declares the prototypes and turns a
non-zero status into ``RuntimeError(idisp_last_error())`` -- the same exception type the
reference's ``AT_ASSERTM`` / ``AT_ERROR`` / ``THCudaCheck`` surface as
(disprcnn/csrc/cuda/ROIAlign_cuda.cu:263-264,297; csrc/ROIAlign.h:21,44).
There is deliberately no fallback: if the shared object is missing the import of any op fails.
"""
import ctypes
import glob
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, 'csrc')
LIB_DIR = os.path.join(_HERE, 'lib')
LIB_PATH = os.path.join(LIB_DIR, 'libidisp.so')
INCLUDE = os.path.join(os.path.dirname(_HERE), 'include')

NVCC_COMPILE_FLAGS = ['-std=c++17', '-O3', '-lineinfo', '-gencode', 'arch=compute_100a,code=sm_100a', '-Xcompiler', '-fPIC']
NVCC_COMPILE_FLAGS += os.environ.get('IDISP_NVCC_EXTRA', '').split()   # e.g. -DIDISP_MRG=0 for an A/B build
NVCC_LINK_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-Xcompiler', '-fPIC', '-shared']
NVCC_FLAGS = NVCC_COMPILE_FLAGS + ['-shared']

PREC_FP32, PREC_BF16, PREC_FP16, PREC_FP16X2 = 0, 1, 2, 3
CONV_S1, CONV_S2, DECONV_S2 = 0, 1, 2

_lib = None


def _sources():
    return sorted(glob.glob(os.path.join(CSRC, '*.cu')))


def _headers():
    return glob.glob(os.path.join(CSRC, '*.cuh')) + glob.glob(os.path.join(INCLUDE, '*.h'))


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in _sources() + _headers())


def build(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a into disprcnn_b200/lib/libidisp.so (nvcc cross-compiles without a GPU).

    One object per source (lib/obj/*.o, compiled in parallel, only the stale ones), then one link."""
    if not force and not _stale():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor
    obj_dir = os.path.join(LIB_DIR, 'obj')
    os.makedirs(obj_dir, exist_ok=True)
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    hdr_t = max([os.path.getmtime(h) for h in _headers()] + [os.path.getmtime(os.path.abspath(__file__))])
    jobs, objs = [], []
    for src in _sources():
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + '.o')
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            jobs.append([nvcc] + NVCC_COMPILE_FLAGS + ['-c', src, '-o', obj])

    def run(cmd):
        if verbose:
            print(' '.join(cmd))
        return subprocess.run(cmd, capture_output=True, text=True)
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        for r in ex.map(run, jobs):
            if r.returncode != 0:
                raise RuntimeError('nvcc failed:\n' + r.stdout + r.stderr)
    r = run([nvcc] + NVCC_LINK_FLAGS + ['-o', LIB_PATH] + objs)
    if r.returncode != 0:
        raise RuntimeError('nvcc (link) failed:\n' + r.stdout + r.stderr)
    return LIB_PATH


_c_float_p = ctypes.POINTER(ctypes.c_float)
_vp, _i, _f, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/idisp.h one to one
PROTOTYPES = {
    'idisp_version': (_i, []),
    'idisp_last_error': (ctypes.c_char_p, []),
    'idisp_roi_align_forward': (_i, [_vp, _i, _i, _i, _i, _vp, _i, _f, _i, _i, _i, _vp, _vp, _vp, _vp]),
    'idisp_roi_align_backward': (_i, [_vp, _vp, _i, _f, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    'idisp_stereo_rois': (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    'idisp_roi_disparity_paste': (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _vp, _i, _i, _vp, _vp]),
    'idisp_roi_depth_paste': (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    'idisp_roi_points_count': (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _f, _i, _vp, _vp]),
    'idisp_roi_points_choice': (_i, [_i, _i, _vp]),
    'idisp_roi_points_gather': (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _f, _i, _vp, _vp, _i, _f, _vp, _vp, _vp, _vp, _vp]),
    'idisp_cost_volume': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    'idisp_conv3d': (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    'idisp_softargmin': (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    'idisp_plan_create': (_i, [_i, _i, _i, _i, ctypes.POINTER(_vp)]),
    'idisp_plan_destroy': (None, [_vp]),
    'idisp_plan_set_tensor': (_i, [_vp, ctypes.c_char_p, _vp, _sz]),
    'idisp_plan_finalize': (_i, [_vp, _vp]),
    'idisp_plan_workspace_bytes': (_sz, [_vp, _i, _i, _i]),
    'idisp_plan_range_exceeded': (_i, [_vp, ctypes.POINTER(ctypes.c_int), _vp]),
    'idisp_plan_forward': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp, _vp]),
    'idisp_plan_forward_host': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'idisp_plan_forward_host_async': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, ctypes.POINTER(ctypes.c_ulonglong)]),
    'idisp_plan_host_wait': (_i, [_vp, ctypes.c_ulonglong]),
    'idisp_plan_get_logits': (_i, [_vp, _vp, _vp]),
    'idisp_plan_launches_per_forward': (_i, [_vp]),
    'idisp_plan_graph_stats': (_i, [_vp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    'idisp_plan_enable_timing': (_i, [_vp, _i]),
    'idisp_plan_get_timing': (_i, [_vp, _vp, _vp, _i]),
    'idisp_extractor_create': (_i, [ctypes.POINTER(_vp)]),
    'idisp_extractor_destroy': (None, [_vp]),
    'idisp_extractor_set_tensor': (_i, [_vp, ctypes.c_char_p, _vp, _sz]),
    'idisp_extractor_finalize': (_i, [_vp, _vp]),
    'idisp_extractor_workspace_bytes': (_sz, [_vp, _i, _i, _i]),
    'idisp_extractor_forward': (_i, [_vp, _vp, _i, _i, _i, _vp, _sz, _vp, _vp]),
    'idisp_extractor_launches_per_forward': (_i, [_vp]),
    'idisp_extractor_set_precision': (_i, [_vp, _i]),
    'idisp_extractor_range_exceeded': (_i, [_vp, ctypes.POINTER(ctypes.c_int), _vp]),
    'idisp_debug_fused_cost_volume': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
}


def load():
    """Return the loaded library (ctypes.CDLL); raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} is missing: the CUDA library has not been built '
            '(run `python -c "import __graft_entry__ as g; g.build()"`). There is no CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().idisp_last_error().decode()


class Unsupported(RuntimeError):
    """IDISP_ERR_UNSUPPORTED (status 3): the selected precision mode does not cover this shape."""


def check(rc):
    if rc != 0:
        raise (Unsupported if rc == 3 else RuntimeError)(f'libidisp: {last_error()} (status {rc})')


def ptr(t):
    """Device/host address of a torch tensor (or None)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError('disprcnn_b200: this op has no CPU path (sm_100a CUDA only); got a CPU tensor')
