"""CPU-side checks of the 3-pass split-tf32 DCN mode (MREFSR_DCN_TF32X3 / the MREFSR_DCN_X3 layout flag): the header,
the Python constants, the workspace sizes it asks for, and the argument checks that run before any CUDA call."""
import ctypes
import os
import re

import pytest

from mrefsr_b200 import _lib
from mrefsr_b200 import dcn as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = ctypes.c_void_p(4096)      # never dereferenced: every call below fails its host-side checks first


def _header_value(name):
    text = open(os.path.join(ROOT, 'include', 'mrefsr_b200.h')).read()
    return int(re.search(r'\b%s\s*=\s*(\d+)' % name, text).group(1))


def _align(n):
    return (n + 1023) // 1024 * 1024


def test_mode_and_flag_values():
    assert _header_value('MREFSR_DCN_TF32X3') == D.DCN_TF32X3 == 3
    assert _header_value('MREFSR_DCN_X3') == D._FLAG_X3 == 8
    assert D._MODES['tf32x3'] == 3
    # the other modes keep their values
    assert (_header_value('MREFSR_DCN_AUTO'), _header_value('MREFSR_DCN_FP32'), _header_value('MREFSR_DCN_TF32')) == (0, 1, 2)
    lib = _lib.lib()
    for sym in ('mrefsr_dcn_pack_weights_x3', 'mrefsr_gemm_tf32x3_nt'):
        assert hasattr(lib, sym) and sym in _lib.SIGNATURES


def test_set_default_mode_accepts_tf32x3():
    try:
        D.set_default_mode('tf32x3')
        assert D._default_mode == D.DCN_TF32X3
    finally:
        D.set_default_mode('auto')
    assert D._default_mode == D.DCN_AUTO


@pytest.mark.parametrize('shape', [(2, 64, 20, 24, 64, 8), (1, 256, 10, 12, 256, 8), (3, 32, 7, 5, 96, 2)])
def test_forward_workspace_counts_the_lo_weights(shape):
    b, c, h, w, co, dg = shape
    ws = _lib.lib().mrefsr_dcn_workspace_bytes
    tf32 = ws(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg, D.DCN_TF32, 0)
    x3 = ws(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg, D.DCN_TF32X3, 0)
    assert tf32 == _align(b * c * h * w * 4) + _align(co * c * 9 * 4) + 1024
    assert x3 == _align(b * c * h * w * 4) + _align(2 * co * c * 9 * 4) + 1024
    # ineligible shapes get no tcgen05 workspace in either mode (they raise in both)
    assert ws(1, 8, 6, 6, 8, 3, 3, 1, 1, 1, 1, 1, 1, 1, 2, D.DCN_TF32X3, 0) == 1024


@pytest.mark.parametrize('shape', [(20, 64, 160, 160, 64, 8, 12), (40, 128, 80, 80, 128, 8, 24),
                                   (60, 256, 40, 40, 256, 8, 48), (2, 32, 10, 12, 32, 8, 2)])
def test_backward_workspace_counts_the_lo_planes(shape):
    """The 3-pass backward adds the lo planes of the GEMM operands (columns chunk, both copies of grad_output, W^T) and
    keeps its three chunk tensors within the 2 GiB the two of the tf32 mode may take: the training shapes then run
    in chunks of 12, 24 and 48 samples instead of 18, 36 and 60."""
    b, c, h, w, co, dg, nb_x3 = shape
    k, p = 9, h * w
    per = c * k * p * 4
    nb_tf32 = max(1, min(b, (1024 << 20) // per))
    assert max(1, min(b, ((2048 << 20) // 3) // per)) == nb_x3
    ws = _lib.lib().mrefsr_dcn_workspace_bytes

    def expect(nb, x3):
        buf, got, gwt = _align(nb * per), _align(b * co * p * 4), _align(co * c * k * 4)
        base = 2 * buf + _align(b * c * h * w * 4) + 2 * got + 2 * gwt + _align(32 * co * c * k * 4) + 1024
        return base + (buf + 2 * got + gwt if x3 else 0)
    assert ws(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg, D.DCN_TF32, 1) == expect(nb_tf32, False)
    assert ws(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg, D.DCN_TF32X3, 1) == expect(nb_x3, True)


def _fused_call(name, flags, c=64, dg=8):
    lib = _lib.lib()
    common = (FAKE, FAKE, None, FAKE, FAKE, 4)
    if name == 'ex':
        return lib.mrefsr_dynagg_dcn_forward_ex(*common, FAKE, 2, c, 16, 16, c, dg, 0, flags, 1.0, FAKE, 1 << 30, None)
    arr = (ctypes.c_void_p * 1)(4096)
    if name == 'multi':
        return lib.mrefsr_dynagg_dcn_forward_multi(*common, ctypes.cast(arr, ctypes.c_void_p), 1, 0, 0, 0, 2, c, 16, 16, c,
                                                   dg, 0, flags, 1.0, FAKE, 1 << 30, None)
    return lib.mrefsr_dynagg_dcn_forward_slabs(*common, ctypes.cast(arr, ctypes.c_void_p), 1, 16, 0, 0, 0, 2, c, 16, 16, c,
                                               dg, 0, flags, 1.0, FAKE, 1 << 30, None)


@pytest.mark.parametrize('name', ['ex', 'multi', 'slabs'])
def test_fused_entry_points_check_the_flags_first(name):
    lib = _lib.lib()
    for bad in (16, 8 | 32, 0x100):
        assert _fused_call(name, bad) < 0
        assert b'flags' in lib.mrefsr_last_error(), (name, bad)
    # the X3 flag itself passes the flag check: an ineligible shape (8 channels) then fails the shape check
    assert _fused_call(name, 8 | 4, c=8, dg=1) < 0
    msg = lib.mrefsr_last_error()
    assert b'flags' not in msg and b'needs' in msg, msg


def test_x3_forward_and_packing_reject_bad_shapes_without_a_gpu():
    lib = _lib.lib()
    # operator entry point, mode 3: an ineligible shape (C % 32 != 0) is refused before any launch
    rc = lib.mrefsr_modulated_deform_conv_forward(FAKE, FAKE, None, FAKE, FAKE, FAKE, 1, 8, 6, 6, 8, 3, 3, 1, 1, 1, 1, 1,
                                                  1, 1, 2, 0, D.DCN_TF32X3, FAKE, 1 << 20, None)
    assert rc < 0 and b'tcgen05 path needs' in lib.mrefsr_last_error()
    # an unknown mode is refused as before
    rc = lib.mrefsr_modulated_deform_conv_forward(FAKE, FAKE, None, FAKE, FAKE, FAKE, 1, 64, 6, 6, 64, 3, 3, 1, 1, 1, 1,
                                                  1, 1, 1, 8, 0, 4, FAKE, 1 << 20, None)
    assert rc < 0 and b'unknown mode' in lib.mrefsr_last_error()
    # the 3-pass packing needs whole 16-channel slabs
    assert lib.mrefsr_dcn_pack_weights_x3(FAKE, FAKE, 32, 24, 9, None) < 0
    assert b'16' in lib.mrefsr_last_error()
    assert lib.mrefsr_dcn_pack_weights_x3(None, FAKE, 32, 32, 9, None) < 0


def test_x3_gemm_entry_checks_its_operands():
    lib = _lib.lib()

    def call(a_hi, a_lo, b_hi, b_lo, lda=64, splits=1, reduce=0):      # 64 x 64 x 64, one batch item
        return lib.mrefsr_gemm_tf32x3_nt(a_hi, a_lo, lda, 0, b_hi, b_lo, 64, 64 * 64, FAKE, 64, 64 * 64, 64, 64, 64, 1,
                                         reduce, splits, None)
    assert call(FAKE, None, FAKE, FAKE) < 0 and b'null' in lib.mrefsr_last_error()
    assert call(FAKE, FAKE, FAKE, None) < 0
    assert call(FAKE, FAKE, FAKE, FAKE, reduce=1, splits=0) < 0 and b'splits' in lib.mrefsr_last_error()
    assert call(FAKE, ctypes.c_void_p(4100), FAKE, FAKE) < 0 and b'aligned' in lib.mrefsr_last_error()
    assert call(FAKE, FAKE, FAKE, FAKE, lda=63) < 0 and b'pitches' in lib.mrefsr_last_error()
