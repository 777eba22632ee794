"""ctypes binding of libmrefsr_b200.so (the C ABI declared in include/mrefsr_b200.h).

There is no CPU fallback: if the library is missing, or a tensor is not on a CUDA device, the
ops raise.  Build the library with ``python -m mrefsr_b200.build`` (or ``__graft_entry__.build()``).
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('MREFSR_LIB') or os.path.join(_HERE, 'lib', 'libmrefsr_b200.so')   # MREFSR_LIB: tuning builds

c_int, c_size_t, c_void_p = ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p

# symbol -> (restype, argtypes); mirrors include/mrefsr_b200.h one to one
_I = c_int
_P = c_void_p
SIGNATURES = {
    'mrefsr_abi_version': (c_int, []),
    'mrefsr_last_error': (ctypes.c_char_p, []),
    'mrefsr_sm_count': (c_int, []),
    'mrefsr_match_workspace_bytes': (c_size_t, [_I] * 8),
    'mrefsr_match_plan': (c_int, [_I] * 9 + [_P]),
    'mrefsr_feature_match_batched': (c_int, [_P, _P] + [_I] * 15 + [_P, _P, _P, c_size_t, _P]),
    'mrefsr_pre_offsets': (c_int, [_P, _I, _I, _I, _P, _P, _P, _P]),
    'mrefsr_dcn_workspace_bytes': (c_size_t, [_I] * 17),
    'mrefsr_dcn_tile_plan': (c_int, [_I, _I, _I, _P, _P, c_size_t]),
    'mrefsr_modulated_deform_conv_forward': (c_int, [_P] * 6 + [_I] * 17 + [_P, c_size_t, _P]),
    'mrefsr_modulated_deform_conv_backward': (c_int, [_P] * 10 + [_I] * 17 + [_P, c_size_t, _P]),
    'mrefsr_gemm_tf32_nt': (c_int, [_P, _I, ctypes.c_longlong, _P, _I, ctypes.c_longlong, _P, _I, ctypes.c_longlong,
                                    _I, _I, _I, _I, _I, _I, _P]),
    'mrefsr_gemm_tf32x3_nt': (c_int, [_P, _P, _I, ctypes.c_longlong, _P, _P, _I, ctypes.c_longlong, _P, _I,
                                      ctypes.c_longlong, _I, _I, _I, _I, _I, _I, _P]),
    'mrefsr_dcn_pack_weights': (c_int, [_P, _P, _I, _I, _I, _P]),
    'mrefsr_dcn_pack_weights_x3': (c_int, [_P, _P, _I, _I, _I, _P]),
    'mrefsr_dynagg_dcn_forward': (c_int, [_P] * 5 + [_I] + [_P] + [_I] * 7 + [_P, c_size_t, _P]),
    'mrefsr_dynagg_dcn_forward_multi': (c_int, [_P] * 5 + [_I] + [_P] + [_I] * 12 + [ctypes.c_float, _P, c_size_t, _P]),
    'mrefsr_dynagg_dcn_forward_slabs': (c_int, [_P] * 5 + [_I] + [_P] + [_I] * 13 + [ctypes.c_float, _P, c_size_t, _P]),
    'mrefsr_dynagg_dcn_forward_ex': (c_int, [_P] * 5 + [_I] + [_P] + [_I] * 8 + [ctypes.c_float, _P, c_size_t, _P]),
    'mrefsr_dynagg_dcn_backward': (c_int, [_P] * 4 + [_I] + [_P] * 5 + [_I] * 9 + [_P, c_size_t, _P]),
    'mrefsr_dynagg_offsets': (c_int, [_P] * 5 + [_I] * 5 + [_P]),
    'mrefsr_dynagg_offsets_backward': (c_int, [_P] * 4 + [_I] * 5 + [_P]),
    'mrefsr_bias_act': (c_int, [_P, _P, _P, _I, _P, _I, _I, _I, _I, _I, _I, _I, ctypes.c_float, ctypes.c_float, _P]),
    'mrefsr_bias_act_train_supported': (c_int, [_I, _I]),
    'mrefsr_bias_act_train_blocks': (c_int, []),
    'mrefsr_bias_act_train_forward': (c_int, [_P, _P, _P, ctypes.c_longlong, _I, _I, _I, ctypes.c_float, ctypes.c_float, _P]),
    'mrefsr_bias_act_train_backward': (c_int, [_P, _P, _P, _P, _P, ctypes.c_longlong, _I, _I, _I, ctypes.c_float,
                                               ctypes.c_float, _P]),
    'mrefsr_maxpool2x2_nhwc': (c_int, [_P, _P, _I, _I, _I, _I, _P]),
    'mrefsr_layout_convert': (c_int, [_P, _P, _P, _I, _I, _I, _I, _P]),
    'mrefsr_layout_convert_bf16': (c_int, [_P, _P, _I, _I, _I, _I, _P]),
    'mrefsr_layout_convert_bf16_act': (c_int, [_P, _P, _P, ctypes.c_float, _I, _I, _I, _I, _P]),
    'mrefsr_attn_modulate': (c_int, [_P] * 5 + [_I] * 4 + [_P]),
    'mrefsr_mrapa_attention_forward': (c_int, [_P] * 5 + [_I] * 6 + [_P]),
    'mrefsr_mrapa_attention_forward_bf16': (c_int, [_P] * 4 + [_I] * 6 + [_P]),
    'mrefsr_mrapa_attention_nhwc': (c_int, [_P] * 7 + [_I, _P, _I, ctypes.c_float, _P] + [_I] * 6 + [_P]),
    'mrefsr_mrapa_attention_backward': (c_int, [_P] * 8 + [_I] * 6 + [_P]),
    'mrefsr_feature_match_batched_host': (c_int, [_P, _P] + [_I] * 15 + [_P, _P, _P]),
    'mrefsr_modulated_deform_conv_forward_host': (c_int, [_P] * 6 + [_I] * 17 + [_P]),
    'mrefsr_mrapa_attention_forward_host': (c_int, [_P] * 4 + [_I] * 6 + [_P]),
    'mrefsr_arena_release': (None, []),
    'mrefsr_launch_count': (ctypes.c_ulonglong, []),
    'mrefsr_timing_enable': (None, [_I]),
    'mrefsr_timing_read': (c_int, [_P, _P, _I]),
}

_lib = None
_lock = threading.Lock()


def lib():
    """The loaded library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        'mrefsr_b200: %s is missing -- build it with `python -m mrefsr_b200.build`. '
                        'There is no CPU / PyTorch fallback for these ops.' % LIB_PATH)
                handle = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().mrefsr_last_error()
        raise RuntimeError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else '?'))


def ptr(t):
    return None if t is None else c_void_p(t.data_ptr())


def stream_ptr(device=None):
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    """Mirror of the reference boundary: CPU tensors are an error
    (basicsr/ops/dcn/deform_conv.py:143-144, deform_conv_ext.cpp:124)."""
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NotImplementedError('mrefsr_b200 ops are CUDA-only (got a %s tensor); there is no CPU path'
                                      % t.device.type)


_workspaces = {}


def workspace(nbytes, device):
    """Per-(device, stream) scratch buffer, grown on demand, 1024-byte aligned.
    Reuse is safe because every consumer runs in stream order on the stream it was handed out for."""
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    buf = _workspaces.get(key)
    need = int(nbytes) + 1024
    if buf is None or buf.numel() < need:
        buf = torch.empty(max(need, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    base = buf.data_ptr()
    aligned = (base + 1023) // 1024 * 1024
    return c_void_p(aligned), buf.numel() - (aligned - base)


def launch_count():
    return int(lib().mrefsr_launch_count())


KERNEL_IDS = ('match_main', 'match_prep', 'dcn_fwd', 'dcn_aux', 'fusion_fwd', 'glue')


def timing_enable(on=True):
    lib().mrefsr_timing_enable(int(bool(on)))


def timing_read():
    """{kernel: (total_ms, launches)} accumulated since the last read (synchronises the recorded events)."""
    n = len(KERNEL_IDS)
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_ulonglong * n)()
    check(lib().mrefsr_timing_read(ctypes.cast(ms, c_void_p), ctypes.cast(cnt, c_void_p), n), 'mrefsr_timing_read')
    return {k: (ms[i], int(cnt[i])) for i, k in enumerate(KERNEL_IDS)}
