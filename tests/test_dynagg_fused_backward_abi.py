"""CPU-side checks of the fused DynAgg backward (mrefsr_dynagg_dcn_backward): the symbol and its header constants, the
argument checks that return a negative code and a message before any CUDA call, and the workspace size it asks for."""
import ctypes
import os
import re

import pytest

from mrefsr_b200 import _lib
from mrefsr_b200 import dcn as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = ctypes.c_void_p(4096)      # never dereferenced: every call below fails its host-side checks first


def _header():
    return open(os.path.join(ROOT, 'include', 'mrefsr_b200.h')).read()


def _call(input=FAKE, weight=FAKE, conv_out=FAKE, max_idx=FAKE, flow_scale=2, grad_output=FAKE, grad_input=FAKE,
          grad_weight=FAKE, grad_bias=FAKE, grad_conv_out=FAKE, shape=(2, 64, 16, 16, 64, 8), with_bias=1, flags=0,
          mode=D.DCN_TF32, workspace=FAKE, workspace_bytes=0):
    b, c, h, w, co, dg = shape
    return _lib.lib().mrefsr_dynagg_dcn_backward(input, weight, conv_out, max_idx, flow_scale, grad_output, grad_input,
                                                 grad_weight, grad_bias, grad_conv_out, b, c, h, w, co, dg, with_bias,
                                                 flags, mode, workspace, workspace_bytes, None)


def _error():
    return _lib.lib().mrefsr_last_error().decode()


def test_symbol_and_header_constants():
    text = _header()
    assert 'MREFSR_API int mrefsr_dynagg_dcn_backward(' in text
    assert re.search(r'\bMREFSR_ABI_VERSION\s+1\b', text)
    for name, value in (('MREFSR_DCN_IN_NHWC', 1), ('MREFSR_DCN_TF32', 2), ('MREFSR_DCN_TF32X3', 3),
                        ('MREFSR_DCN_FP32', 1)):
        assert int(re.search(r'\b%s\s*=\s*(\d+)' % name, text).group(1)) == value
    assert hasattr(_lib.lib(), 'mrefsr_dynagg_dcn_backward') and 'mrefsr_dynagg_dcn_backward' in _lib.SIGNATURES
    assert _lib.lib().mrefsr_abi_version() == 1


@pytest.mark.parametrize('arg', ['input', 'weight', 'conv_out', 'max_idx', 'grad_output'])
def test_null_pointers_are_refused(arg):
    assert _call(**{arg: None}) == -1 and 'null pointer' in _error()


def test_argument_errors_come_back_before_device_work():
    assert _call(with_bias=1, grad_bias=None) == -1 and 'grad_bias' in _error()
    assert _call(flow_scale=3) == -1 and 'multiple of the flow scale 3' in _error()       # 16 % 3 != 0
    assert _call(flow_scale=0) == -1 and 'flow scale' in _error()
    assert _call(flow_scale=8) == -1 and 'grid too small' in _error()                     # 16 / 8 - 2 = 0 rows
    assert _call(flags=2) == -1 and 'layout flags' in _error()                             # OUT_NHWC: forward only
    assert _call(flags=8) == -1 and 'layout flags' in _error()
    assert _call(flags=1, input=ctypes.c_void_p(4096 + 16)) == -1 and 'aligned' in _error()
    assert _call(mode=7) == -1 and 'unknown mode' in _error()


def test_fp32_mode_and_ineligible_shapes_are_unsupported():
    assert _call(mode=D.DCN_FP32) == -2 and 'fp32' in _error()
    for shape in ((2, 8, 16, 16, 8, 1), (2, 64, 16, 16, 48, 8), (2, 64, 16, 16, 64, 16), (2, 64, 16, 16, 512, 8)):
        assert _call(shape=shape) == -2 and 'needs' in _error(), shape


@pytest.mark.parametrize('shape', [(60, 256, 40, 40, 256, 8, 1), (40, 128, 80, 80, 128, 8, 2),
                                   (20, 64, 160, 160, 64, 8, 4), (2, 64, 76, 76, 64, 2, 1)])
@pytest.mark.parametrize('mode', [D.DCN_AUTO, D.DCN_TF32, D.DCN_TF32X3])
def test_workspace_size_covers_the_entry(shape, mode):
    """The size the entry point asks for (reported when it gets none) is within mrefsr_dcn_workspace_bytes(...,
    backward=1) for the resolved mode: the fused backward needs no sizing function of its own."""
    b, c, h, w, co, dg, s = shape
    resolved = D.DCN_TF32 if mode == D.DCN_AUTO else mode
    have = _lib.lib().mrefsr_dcn_workspace_bytes(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg, resolved, 1)
    assert _call(shape=shape[:6], flow_scale=s, mode=mode, workspace_bytes=0) == -3
    m = re.search(r'workspace too small \(0 < (\d+)\)', _error())
    assert m, _error()
    assert 0 < int(m.group(1)) <= have
