"""CPU: the C-ABI library loads, exports every symbol include/idisp.h declares, validates arguments
without touching a GPU, and the Python mirror keeps the reference's API surface."""
import ctypes
import inspect
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'idisp.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(idisp_[a-z0-9_]+)\s*\(', text)))


def test_header_symbols_are_exported(built_lib):
    from disprcnn_b200 import _lib
    names = _declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(built_lib, n), f'{n} declared in include/idisp.h but not exported by libidisp.so'
    assert sorted(_lib.PROTOTYPES) == names  # the ctypes table binds exactly the header
    assert built_lib.idisp_version() == 2


def test_argument_validation_without_gpu(built_lib):
    from disprcnn_b200 import _lib
    lib = built_lib
    h = ctypes.c_void_p()
    assert lib.idisp_plan_create(32, -48, 48, 0, ctypes.byref(h)) == 0 and h.value
    assert lib.idisp_plan_forward(h, None, None, 1, 16, 16, 64, 64, None, 0, None, None) == 4  # not finalised
    assert 'finalise' in _lib.last_error()
    assert lib.idisp_plan_finalize(h, None) == 4 and "dres0.0.0.weight" in _lib.last_error()  # missing weights named
    assert lib.idisp_plan_workspace_bytes(h, 2, 16, 16) > 0
    lib.idisp_plan_destroy(h)
    bad = ctypes.c_void_p()
    assert lib.idisp_plan_create(32, -46, 48, 0, ctypes.byref(bad)) == 1 and 'multiples of 4' in _lib.last_error()
    assert lib.idisp_plan_create(32, -48, 48, 7, ctypes.byref(bad)) == 1 and 'precision' in _lib.last_error()
    assert lib.idisp_plan_create(32, 0, 24, 0, ctypes.byref(bad)) == 1  # D=6 not a multiple of 4
    assert lib.idisp_cost_volume(None, None, 1, 32, 0, 16, -16, 16, None, None) == 1
    assert lib.idisp_roi_align_forward(None, 1, 3, 8, 8, None, 2, 1.0, 0, 7, 0, None, None, None, None) == 1
    assert lib.idisp_roi_align_forward(None, 1, 3, 8, 8, None, 0, 1.0, 7, 7, 0, None, None, None, None) == 0  # R=0 no-op
    assert lib.idisp_roi_align_backward(None, None, 0, 1.0, 7, 7, 1, 3, 8, 8, 0, None, None) == 3
    assert lib.idisp_stereo_rois(None, None, None, 0, 1242, 375, None, 0, None, None, None, None) == 0           # R=0 no-op
    assert lib.idisp_stereo_rois(None, None, None, 2, 1242, 375, None, 0, None, None, None, None) == 1 and 'NULL' in _lib.last_error()
    assert lib.idisp_stereo_rois(None, None, None, 2, 0, 375, None, 0, None, None, None, None) == 1
    assert lib.idisp_softargmin(None, 1, 8, 4, 4, 0, 4, 16, 16, None, None) == 1  # Dfull < D
    assert lib.idisp_conv3d(None, 1, 12, 4, 4, 4, None, 32, 0, None, None, None, 0, 0, None, None) == 1  # Cin % 8


def test_python_api_mirrors_reference(built_lib):
    from disprcnn_b200.layers import ROIAlign, roi_align
    from disprcnn_b200.modeling.psmnet import stackhourglass, submodule
    # constructor / forward signatures of disprcnn/layers/roi_align.py:52-65
    assert list(inspect.signature(ROIAlign.__init__).parameters)[1:] == ['output_size', 'spatial_scale', 'sampling_ratio']
    assert list(inspect.signature(ROIAlign.forward).parameters)[1:] == ['input', 'rois', 'spatial_scale']
    assert repr(ROIAlign((224, 224), 1.0, 0)) == 'ROIAlign(output_size=(224, 224), spatial_scale=1.0, sampling_ratio=0)'
    # PSMNet positional signature of stackhourglass.py:55-58
    params = list(inspect.signature(stackhourglass.PSMNet.__init__).parameters)[1:9]
    assert params == ['maxdisp', 'mindisp', 'input_size', 'is_module', 'feature_level',
                      'single_modal_weight_average', 'conv_layers', 'use_disparity_regression']
    m = stackhourglass.PSMNet(48, -48)
    sd = m.state_dict()
    assert len(sd) == 514 and sum(not k.startswith('feature_extraction') for k in sd) == 153
    assert tuple(sd['dres0.0.0.weight'].shape) == (32, 64, 3, 3, 3)
    assert tuple(sd['dres2.conv5.0.weight'].shape) == (64, 64, 3, 3, 3)
    assert tuple(sd['dres3.conv6.0.weight'].shape) == (64, 32, 3, 3, 3)  # ConvTranspose layout [Cin,Cout,...]
    assert tuple(sd['classif1.2.weight'].shape) == (1, 32, 3, 3, 3)
    for name in ('convbn_3d', 'disparityregression', 'feature_extraction', 'convbn', 'BasicBlock'):
        assert hasattr(submodule, name)
    # no CPU fallback: CPU tensors are refused loudly
    m.eval()
    with pytest.raises(RuntimeError, match='no CPU path'):
        m.forward_features(torch.zeros(1, 32, 16, 16), torch.zeros(1, 32, 16, 16))
    with pytest.raises(RuntimeError, match='no CPU path'):
        roi_align(torch.zeros(1, 3, 8, 8), torch.zeros(1, 5), (7, 7), 1.0, 0)
    with pytest.raises(RuntimeError, match='inference-only'):
        stackhourglass.PSMNet(48, -48).train().forward_features(torch.zeros(1, 32, 16, 16), torch.zeros(1, 32, 16, 16))
    p = torch.softmax(torch.randn(1, 8, 2, 2), 1)
    assert torch.allclose(submodule.disparityregression(p, 8, 0), (p * torch.arange(8.).view(1, 8, 1, 1)).sum(1))


def test_install_aliases_reference_import_paths(built_lib):
    import sys
    import disprcnn_b200
    saved = {k: sys.modules.get(k) for k in ('disprcnn.layers.roi_align', 'disprcnn.modeling.psmnet.stackhourglass',
                                             'disprcnn.modeling.psmnet.submodule')}
    try:
        disprcnn_b200.install(inference_only=True)
        from disprcnn_b200.modeling.psmnet import stackhourglass
        assert sys.modules['disprcnn.modeling.psmnet.stackhourglass'] is stackhourglass
        assert sys.modules['disprcnn.layers.roi_align'].ROIAlign.__module__ == 'disprcnn_b200.layers.roi_align'
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_psmnet_default_precision_picks_the_parity_grade_mode_the_shape_allows():
    """precision='auto' (the default a drop-in caller gets): split-precision tensor-core kernels where they apply, fp32 FFMA
    otherwise -- never a one-word mode, which would miss the 1e-3 bar."""
    from disprcnn_b200.modeling.psmnet.stackhourglass import PSMNet
    assert PSMNet(96, -96).precision == 'auto'
    assert PSMNet(96, -96).effective_precision(112, 112) == 'fp16x2'                       # BASELINE configs[1]
    assert PSMNet(48, -48).effective_precision(56, 56) == 'fp16x2'                         # the live KITTI shape
    assert PSMNet(48, -48, feature_channels=16).effective_precision(64, 64) == 'fp16x2'    # configs[0]
    assert PSMNet(16, -24, feature_channels=32).effective_precision(16, 16) == 'fp32'      # D = 10: not a multiple of 4
    assert PSMNet(48, -48, feature_channels=8).effective_precision(32, 32) == 'fp32'       # C = 8
    assert PSMNet(48, -48, precision='bf16').effective_precision(56, 56) == 'bf16'         # explicit choice is kept
    import pytest
    with pytest.raises(ValueError):
        PSMNet(48, -48, precision='int8')


# A minimal ``disprcnn`` package tree with the import pattern install() has to serve (SURVEY.md 8(b)): layer modules that read
# ``disprcnn._C`` at import time, a layers package re-exporting ROIAlign, and consumers importing PSMNet and ROIAlign by the
# reference's names.  Only the modules install() does not replace are written out; the rest must come from disprcnn_b200.
_STAND_IN_TREE = {
    'disprcnn/__init__.py': '',
    'disprcnn/layers/__init__.py': 'from .nms import nms\nfrom .roi_pool import roi_pool\nfrom .roi_align import ROIAlign, roi_align\n'
                                   '__all__ = ["nms", "roi_pool", "ROIAlign", "roi_align"]\n',
    'disprcnn/layers/nms.py': 'from disprcnn import _C\nnms = _C.nms\n',
    'disprcnn/layers/roi_pool.py': 'from disprcnn import _C\nroi_pool = _C.roi_pool_forward\n',
    'disprcnn/modeling/__init__.py': '',
    'disprcnn/modeling/poolers.py': 'from torch import nn\nfrom disprcnn.layers import ROIAlign\n\n\n'
                                    'class Pooler(nn.Module):\n'
                                    '    def __init__(self, output_size, scales, sampling_ratio):\n'
                                    '        super().__init__()\n'
                                    '        self.poolers = nn.ModuleList(ROIAlign(output_size, s, sampling_ratio) for s in scales)\n',
    'disprcnn/modeling/psmnet/__init__.py': '',
}


def test_install_routes_a_disprcnn_package_tree_to_this_package(built_lib, tmp_path):
    """After install() a ``disprcnn`` package laid out like the reference's imports: its layer modules get ``disprcnn._C`` (the
    reference's pybind module, which does not build on torch 2.x) from disprcnn_b200._C, and ROIAlign / PSMNet resolve to the
    B200 classes wherever they are imported.  Run in a subprocess: it puts a ``disprcnn`` package on sys.path."""
    import subprocess
    import sys
    for rel, text in _STAND_IN_TREE.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    code = r'''
import sys, warnings
sys.path.insert(0, %r); sys.path.insert(1, %r)
import disprcnn_b200
with warnings.catch_warnings(record=True) as w:
    warnings.simplefilter('always')
    disprcnn_b200.install()
assert any('inference-only' in str(x.message) for x in w), 'install() must say that it is inference-only'
disprcnn_b200.install(inference_only=True)
from disprcnn.layers import ROIAlign, roi_align, nms, roi_pool
assert ROIAlign.__module__ == 'disprcnn_b200.layers.roi_align', ROIAlign.__module__
from disprcnn import _C
import disprcnn_b200._C as shim
assert _C is shim
for name in ('nms', 'roi_align_forward', 'roi_align_backward', 'roi_pool_forward', 'roi_pool_backward',
             'sigmoid_focalloss_forward', 'sigmoid_focalloss_backward'):   # csrc/vision.cpp:7-15
    assert callable(getattr(_C, name)), name
import torch
for fn in (nms, roi_pool, _C.roi_align_backward, _C.roi_pool_forward):
    try:
        fn(torch.zeros(1, 4), torch.zeros(1), 0.5)
    except RuntimeError as e:
        assert 'B200' in str(e)
    else:
        raise AssertionError('detector ops must raise when called')
try:
    _C.roi_align_forward(torch.zeros(1, 3, 8, 8), torch.zeros(1, 5), 1.0, 4, 4, 0)   # CPU tensors: no CPU path
except RuntimeError as e:
    assert 'no CPU path' in str(e)
else:
    raise AssertionError('CPU tensors must raise')
from disprcnn.modeling.psmnet.stackhourglass import PSMNet
assert PSMNet.__module__ == 'disprcnn_b200.modeling.psmnet.stackhourglass'
from disprcnn.modeling.poolers import Pooler   # second ROIAlign consumer
p = Pooler((7, 7), (0.25, 0.125), 2)
assert type(p.poolers[0]).__module__ == 'disprcnn_b200.layers.roi_align'
print('ok')
''' % (ROOT, str(tmp_path))
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith('ok'), r.stdout + r.stderr
