"""Modulated deformable convolution (DCNv2): host-side mirror of basicsr/ops/dcn/deform_conv.py on the sm_100a
kernels of csrc/dcn.cu / csrc/dcn_tc.cu.

Same operator API as the reference (deform_conv.py:121-188, :289-379):
    ModulatedDeformConvFunction.apply(input, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1,
                                      groups=1, deformable_groups=1)
    modulated_deform_conv = ModulatedDeformConvFunction.apply
    ModulatedDeformConv, ModulatedDeformConvPack  (same parameters / state-dict keys / init)
stride / padding / dilation may be ints (basicsr) or pairs (mmcv.ops, see mmcv_ops.py).
DCNv1 (DeformConv, DeformConvPack, deform_conv; deform_conv.py:33-118, :191-286) is exported by the reference
package but unused by MRefSR; it runs on the same kernels with an implicit all-ones mask.
"""
import math

import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable
from torch.nn.modules.utils import _pair, _single

from . import _lib

DCN_AUTO, DCN_FP32, DCN_TF32, DCN_TF32X3 = 0, 1, 2, 3
_MODES = {'auto': DCN_AUTO, 'fp32': DCN_FP32, 'tf32': DCN_TF32, 'tf32x3': DCN_TF32X3}
_default_mode = DCN_AUTO
_FLAG_X3 = 8          # MREFSR_DCN_X3: layout flag of the fused DynAgg entry points


def _mode(mode):
    return _default_mode if mode is None else (_MODES[mode] if isinstance(mode, str) else int(mode))


def set_default_mode(mode):
    """'auto' | 'fp32' (exact, CUDA cores) | 'tf32' (tcgen05) | 'tf32x3' (tcgen05 with 3-pass split-tf32 operands:
    fp32-grade results in the forward and in the backward GEMMs, same shapes as 'tf32', and the fused DynAgg entry
    points follow it too)."""
    global _default_mode
    _default_mode = _mode(mode)


def pack_weight(weight, mode=None):
    """tf32-rounded [Co][tap][C] copy of a DCN weight, the B operand of the tcgen05 kernels (mrefsr_dcn_pack_weights).
    mode (default: the default mode) 'tf32x3': the 3-pass kernels' hi / lo packing [Co][tap][C/16][hi 16 | lo 16]
    (mrefsr_dcn_pack_weights_x3, twice the size), the one `dynagg_dcn_forward` wants while the default mode is 'tf32x3'.
    The forward entry points repack on every call (a few microseconds); a caller whose weights are frozen may pack once
    and hand the result to `dynagg_dcn_forward(..., weight_packed=...)`.  There is deliberately NO implicit cache:
    torch's version counter does not see `weight.data.copy_(...)`-style updates, and a stale packing would be a silent
    wrong answer for a 0.2 % gain."""
    _lib.require_cuda(weight)
    x3 = _mode(mode) == DCN_TF32X3
    w = weight.detach().contiguous().float()
    co, c, kh, kw = w.shape
    packed = torch.empty(co, kh * kw * c * (2 if x3 else 1), dtype=torch.float32, device=w.device)
    fn = 'mrefsr_dcn_pack_weights_x3' if x3 else 'mrefsr_dcn_pack_weights'
    with torch.cuda.device(w.device):
        rc = getattr(_lib.lib(), fn)(_lib.ptr(w), _lib.ptr(packed), co, c, kh * kw, _lib.stream_ptr(w.device))
    _lib.check(rc, fn)
    return packed


def _out_hw(h, w, kh, kw, stride, padding, dilation):
    ho = (h + 2 * padding[0] - (dilation[0] * (kh - 1) + 1)) // stride[0] + 1
    wo = (w + 2 * padding[1] - (dilation[1] * (kw - 1) + 1)) // stride[1] + 1
    return ho, wo


def _check_shapes(input, offset, mask, weight, groups, dg, ho, wo):
    b, c = input.shape[:2]
    co, cg, kh, kw = weight.shape
    if c != cg * groups:
        raise RuntimeError("Input shape and kernel channels won't match: (%d vs %d)." % (c, cg * groups))
    if tuple(offset.shape) != (b, 2 * dg * kh * kw, ho, wo):
        raise RuntimeError('offset shape %s, expected %s' % (tuple(offset.shape), (b, 2 * dg * kh * kw, ho, wo)))
    if mask is not None and tuple(mask.shape) != (b, dg * kh * kw, ho, wo):
        raise RuntimeError('mask shape %s, expected %s' % (tuple(mask.shape), (b, dg * kh * kw, ho, wo)))


def dcn_forward_raw(input, offset, mask, weight, bias, stride, padding, dilation, groups, dg, mode=None):
    """Forward on contiguous fp32 CUDA tensors -> output [B,Co,Ho,Wo] (no autograd).  mask=None: all-ones (DCNv1).
    mode: 'auto' | 'fp32' | 'tf32' | 'tf32x3' (or the C enum value); None: the default mode."""
    lib = _lib.lib()
    b, c, h, w = input.shape
    co, _, kh, kw = weight.shape
    ho, wo = _out_hw(h, w, kh, kw, stride, padding, dilation)
    _check_shapes(input, offset, mask, weight, groups, dg, ho, wo)
    m = _mode(mode)
    out = torch.empty(b, co, ho, wo, dtype=torch.float32, device=input.device)
    with torch.cuda.device(input.device):
        nbytes = lib.mrefsr_dcn_workspace_bytes(b, c, h, w, co, kh, kw, stride[0], stride[1], padding[0], padding[1],
                                                dilation[0], dilation[1], groups, dg, m, 0)
        ws, ws_bytes = _lib.workspace(nbytes, input.device)
        rc = lib.mrefsr_modulated_deform_conv_forward(
            _lib.ptr(input), _lib.ptr(weight), _lib.ptr(bias), _lib.ptr(offset), _lib.ptr(mask), _lib.ptr(out), b, c, h,
            w, co, kh, kw, stride[0], stride[1], padding[0], padding[1], dilation[0], dilation[1], groups, dg,
            int(bias is not None), m, ws, ws_bytes, _lib.stream_ptr(input.device))
    _lib.check(rc, 'mrefsr_modulated_deform_conv_forward')
    return out


def dynagg_dcn_forward_into(input, conv_out, max_idx, flow_scale, weight, bias, deformable_groups, out_ptrs,
                            dst_group, dst_stride, dst_offset, out_slope=1.0, slab_rows=0):
    """Fused DynAgg forward whose epilogue stores straight into several gathered buffers [n, R, Co, H, W] (NCHW
    planes): `out_ptrs` are device addresses of this GPU's and the peers' copies (see parallel.PeerGatherBuffer);
    sample b lands in slot (b // dst_group) * dst_stride + dst_offset + b % dst_group.  Returns nothing: the data is
    in the buffers once the kernel and the caller's cross-GPU barrier have completed.
    slab_rows > 0: pixel-slab routing -- `out_ptrs` are the ranks' buffers IN RANK ORDER, each [n, R, Co, slab_rows, W],
    and output row oy goes to buffer oy // slab_rows only (parallel.PeerSlabBuffer)."""
    import ctypes
    from .trunk import to_nchw
    _lib.require_cuda(input, conv_out, max_idx, weight, bias)
    lib = _lib.lib()
    x = input.float()
    in_cl = x.dim() == 4 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last)
    if not in_cl:
        x = x.contiguous()
    co_, wgt = to_nchw(conv_out.float()), weight.contiguous().float()
    bs = bias.contiguous().float() if bias is not None else None
    mi = max_idx.contiguous()
    b, c, h, w = x.shape
    co, dg = wgt.shape[0], deformable_groups
    if tuple(co_.shape) != (b, 3 * dg * 9, h, w):
        raise RuntimeError('conv_out shape %s, expected %s' % (tuple(co_.shape), (b, 3 * dg * 9, h, w)))
    if mi.dtype != torch.int64 or tuple(mi.shape) != (b, h // flow_scale - 2, w // flow_scale - 2):
        raise RuntimeError('max_idx must be int64 [%d,%d,%d]' % (b, h // flow_scale - 2, w // flow_scale - 2))
    if tuple(wgt.shape[1:]) != (c, 3, 3):
        raise RuntimeError('weight shape %s, expected [Co,%d,3,3]' % (tuple(wgt.shape), c))
    if not 1 <= len(out_ptrs) <= 8:
        raise ValueError('1..8 destination buffers')
    arr = (ctypes.c_void_p * len(out_ptrs))(*[int(p) for p in out_ptrs])
    x3 = _default_mode == DCN_TF32X3
    flags = (1 if in_cl else 0) | (_FLAG_X3 if x3 else 0)
    with torch.cuda.device(x.device):
        nbytes = lib.mrefsr_dcn_workspace_bytes(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg,
                                                DCN_TF32X3 if x3 else DCN_TF32, 0)
        ws, ws_bytes = _lib.workspace(nbytes, x.device)
        if slab_rows:
            if slab_rows * len(out_ptrs) < h:
                raise ValueError('slab_rows * buffers must cover the %d output rows' % h)
            rc = lib.mrefsr_dynagg_dcn_forward_slabs(_lib.ptr(x), _lib.ptr(wgt), _lib.ptr(bs), _lib.ptr(co_), _lib.ptr(mi),
                                                     int(flow_scale), ctypes.cast(arr, ctypes.c_void_p), len(out_ptrs),
                                                     int(slab_rows), int(dst_group), int(dst_stride), int(dst_offset), b, c,
                                                     h, w, co, dg, int(bs is not None), flags, float(out_slope),
                                                     ws, ws_bytes, _lib.stream_ptr(x.device))
        else:
            rc = lib.mrefsr_dynagg_dcn_forward_multi(_lib.ptr(x), _lib.ptr(wgt), _lib.ptr(bs), _lib.ptr(co_), _lib.ptr(mi),
                                                     int(flow_scale), ctypes.cast(arr, ctypes.c_void_p), len(out_ptrs),
                                                     int(dst_group), int(dst_stride), int(dst_offset), b, c, h, w, co, dg,
                                                     int(bs is not None), flags, float(out_slope), ws, ws_bytes,
                                                     _lib.stream_ptr(x.device))
    _lib.check(rc, 'mrefsr_dynagg_dcn_forward_slabs' if slab_rows else 'mrefsr_dynagg_dcn_forward_multi')


def dynagg_dcn_forward(input, conv_out, max_idx, flow_scale, weight, bias, deformable_groups, out_slope=1.0,
                       out_channels_last=None, weight_packed=None):
    """Fused DynAgg forward (no autograd; dynagg.DynAggFusedFunction is its autograd node): DCNv2 (3x3, stride 1, pad 1) whose offsets and masks are
    assembled inside the gather from the raw conv_offset_mask output and the matcher's arg-max map
    (ref_mrapa_restoration_arch.py:45-76 + corres_generation_arch.py:30-47, :70-105 for one scale).
    input [B,C,H,W], conv_out [B,3*dg*9,H,W], max_idx int64 [B,H/s-2,W/s-2] -> [B,Co,H,W].
    A torch.channels_last `input` is consumed as it is (it already is the gather layout); the result is
    channels_last when `out_channels_last` (default: follows the input).  out_slope: leaky-ReLU slope applied to the
    result in the epilogue (1.0 = none).  weight_packed: optional `pack_weight(weight)` (skips the per-call repack).
    While the default mode is 'tf32x3' this runs the 3-pass kernel (fp32-grade) and weight_packed must come from
    `pack_weight(weight, 'tf32x3')`; every other mode runs the tf32 kernel, as this entry point always has."""
    _lib.require_cuda(input, conv_out, max_idx, weight, bias)
    lib = _lib.lib()
    x = input.float()
    in_cl = x.dim() == 4 and not x.is_contiguous() and x.is_contiguous(memory_format=torch.channels_last)
    if not in_cl:
        x = x.contiguous()
    if out_channels_last is None:
        out_channels_last = in_cl
    from .trunk import to_nchw
    co_, wgt = to_nchw(conv_out.float()), weight.contiguous().float()
    bs = bias.contiguous().float() if bias is not None else None
    mi = max_idx.contiguous()
    b, c, h, w = x.shape
    co = wgt.shape[0]
    dg = deformable_groups
    if tuple(co_.shape) != (b, 3 * dg * 9, h, w):
        raise RuntimeError('conv_out shape %s, expected %s' % (tuple(co_.shape), (b, 3 * dg * 9, h, w)))
    if mi.dtype != torch.int64 or tuple(mi.shape) != (b, h // flow_scale - 2, w // flow_scale - 2):
        raise RuntimeError('max_idx must be int64 [%d,%d,%d]' % (b, h // flow_scale - 2, w // flow_scale - 2))
    if tuple(wgt.shape[1:]) != (c, 3, 3):
        raise RuntimeError('weight shape %s, expected [Co,%d,3,3]' % (tuple(wgt.shape), c))
    out = torch.empty(b, co, h, w, dtype=torch.float32, device=x.device,
                      memory_format=torch.channels_last if out_channels_last else torch.contiguous_format)
    x3 = _default_mode == DCN_TF32X3
    flags = (1 if in_cl else 0) | (2 if out_channels_last else 0) | (_FLAG_X3 if x3 else 0)
    if weight_packed is not None:        # pack_weight(weight), made once by a caller whose weights are frozen
        if (tuple(weight_packed.shape) != (co, 9 * c * (2 if x3 else 1)) or weight_packed.dtype != torch.float32 or
                not weight_packed.is_contiguous()):
            raise RuntimeError('weight_packed must be the result of pack_weight(weight%s)' % (", 'tf32x3'" if x3 else ''))
        wgt, flags = weight_packed, flags | 4
    with torch.cuda.device(x.device):
        nbytes = lib.mrefsr_dcn_workspace_bytes(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg,
                                                DCN_TF32X3 if x3 else DCN_TF32, 0)
        ws, ws_bytes = _lib.workspace(nbytes, x.device)
        rc = lib.mrefsr_dynagg_dcn_forward_ex(_lib.ptr(x), _lib.ptr(wgt), _lib.ptr(bs), _lib.ptr(co_), _lib.ptr(mi),
                                              int(flow_scale), _lib.ptr(out), b, c, h, w, co, dg, int(bs is not None),
                                              flags, float(out_slope), ws, ws_bytes, _lib.stream_ptr(x.device))
    _lib.check(rc, 'mrefsr_dynagg_dcn_forward_ex')
    return out


def dynagg_dcn_backward_raw(input, conv_out, max_idx, flow_scale, weight, grad_output, deformable_groups, with_bias,
                            need_input=True, need_conv=True, need_weight=True, mode=None):
    """Backward of `dynagg_dcn_forward` (mrefsr_dynagg_dcn_backward, no autograd) -> (grad_input, grad_conv_out,
    grad_weight, grad_bias); parts not requested (or no bias) are None.  input: the fp32 tensor the forward read (dense
    NCHW or channels_last; grad_input comes back in the same layout); conv_out fp32 NCHW [B,3*dg*9,H,W]; max_idx int64
    [B,H/s-2,W/s-2]; weight fp32 [Co,C,3,3]; grad_output fp32 NCHW [B,Co,H,W].  grad_conv_out = [d offset,
    d mask * mask * (1 - mask)] at conv_out's channels.  mode None: 'tf32x3' while that is the default mode, else 'tf32'
    (the modes the fused forward runs); 'fp32' is refused."""
    from .trunk import is_channels_last
    lib = _lib.lib()
    in_cl = is_channels_last(input)
    b, c, h, w = input.shape
    co, dg = weight.shape[0], deformable_groups
    m = (DCN_TF32X3 if _default_mode == DCN_TF32X3 else DCN_TF32) if mode is None else _mode(mode)
    for name, t in (('input', input), ('conv_out', conv_out), ('weight', weight), ('grad_output', grad_output)):
        if t.dtype != torch.float32 or not (t.is_contiguous() or (t is input and in_cl)):
            raise RuntimeError('%s must be a dense fp32 tensor' % name)
    if tuple(conv_out.shape) != (b, 3 * dg * 9, h, w) or tuple(grad_output.shape) != (b, co, h, w):
        raise RuntimeError('conv_out / grad_output shapes %s / %s, expected %s / %s' % (
            tuple(conv_out.shape), tuple(grad_output.shape), (b, 3 * dg * 9, h, w), (b, co, h, w)))
    if max_idx.dtype != torch.int64 or not max_idx.is_contiguous() or \
            tuple(max_idx.shape) != (b, h // flow_scale - 2, w // flow_scale - 2):
        raise RuntimeError('max_idx must be contiguous int64 [%d,%d,%d]' % (b, h // flow_scale - 2, w // flow_scale - 2))
    if tuple(weight.shape[1:]) != (c, 3, 3):
        raise RuntimeError('weight shape %s, expected [Co,%d,3,3]' % (tuple(weight.shape), c))
    gi = torch.empty_like(input) if need_input else None
    gc = torch.empty_like(conv_out) if need_conv else None
    gw = torch.zeros_like(weight) if need_weight else None
    gb = torch.zeros(co, dtype=torch.float32, device=input.device) if with_bias else None
    with torch.cuda.device(input.device):
        nbytes = lib.mrefsr_dcn_workspace_bytes(b, c, h, w, co, 3, 3, 1, 1, 1, 1, 1, 1, 1, dg,
                                                DCN_TF32 if m == DCN_AUTO else m, 1)
        ws, ws_bytes = _lib.workspace(nbytes, input.device)
        rc = lib.mrefsr_dynagg_dcn_backward(_lib.ptr(input), _lib.ptr(weight), _lib.ptr(conv_out), _lib.ptr(max_idx),
                                            int(flow_scale), _lib.ptr(grad_output), _lib.ptr(gi), _lib.ptr(gw),
                                            _lib.ptr(gb), _lib.ptr(gc), b, c, h, w, co, dg, int(with_bias),
                                            1 if in_cl else 0, m, ws, ws_bytes, _lib.stream_ptr(input.device))
    _lib.check(rc, 'mrefsr_dynagg_dcn_backward')
    return gi, gc, gw, gb


def _nchw(t):
    """dense NCHW fp32 view / copy of an activation (channels-last tensors go through the tiled transpose kernel)."""
    from .trunk import to_nchw_f32
    return to_nchw_f32(t)


class ModulatedDeformConvFunction(Function):

    @staticmethod
    def forward(ctx, input, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1, groups=1,
                deformable_groups=1):
        ctx.stride, ctx.padding, ctx.dilation = _pair(stride), _pair(padding), _pair(dilation)
        ctx.groups = groups
        ctx.deformable_groups = deformable_groups
        ctx.with_bias = bias is not None
        if not input.is_cuda:
            raise NotImplementedError  # same as deform_conv.py:143-144
        _lib.require_cuda(offset, mask, weight, bias)
        ctx.in_dtype = input.dtype
        x, off, msk = (_nchw(t) for t in (input, offset, mask))
        wgt = weight.contiguous().float()
        bs = bias.contiguous().float() if bias is not None else None
        if weight.requires_grad or mask.requires_grad or offset.requires_grad or input.requires_grad:
            ctx.save_for_backward(x, off, msk, wgt)
        out = dcn_forward_raw(x, off, msk, wgt, bs, ctx.stride, ctx.padding, ctx.dilation, groups, deformable_groups)
        return out.to(input.dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        if not grad_output.is_cuda:
            raise NotImplementedError
        x, off, msk, wgt = ctx.saved_tensors
        grad_input, grad_offset, grad_mask, grad_weight, grad_bias = dcn_backward_raw(
            x, off, msk, wgt, _nchw(grad_output), ctx.stride, ctx.padding, ctx.dilation, ctx.groups,
            ctx.deformable_groups, ctx.with_bias, need_input=ctx.needs_input_grad[0])
        dt = ctx.in_dtype
        cast = (lambda t: None if t is None else t.to(dt))
        return (cast(grad_input), cast(grad_offset), cast(grad_mask), cast(grad_weight), cast(grad_bias), None, None,
                None, None, None)

    @staticmethod
    def _infer_shape(ctx, input, weight):
        n = input.size(0)
        kh, kw = weight.shape[2:4]
        ho, wo = _out_hw(input.shape[2], input.shape[3], kh, kw, _pair(ctx.stride), _pair(ctx.padding),
                         _pair(ctx.dilation))
        return n, weight.size(0), ho, wo


modulated_deform_conv = ModulatedDeformConvFunction.apply


def dcn_backward_raw(input, offset, mask, weight, grad_output, stride, padding, dilation, groups, dg, with_bias,
                     need_input=True, need_offset=True, need_weight=True):
    """Backward on contiguous fp32 CUDA tensors -> (grad_input, grad_offset, grad_mask, grad_weight, grad_bias);
    entries that were not requested (or do not exist: mask None, no bias) are None."""
    lib = _lib.lib()
    b, c, h, w = input.shape
    co, _, kh, kw = weight.shape
    gi = torch.empty_like(input) if need_input else None
    go = torch.empty_like(offset) if need_offset else None
    gm = torch.empty_like(mask) if (need_offset and mask is not None) else None
    gw = torch.zeros_like(weight) if need_weight else None
    gb = torch.zeros(co, dtype=torch.float32, device=input.device) if with_bias else None
    s, p, d = stride, padding, dilation
    with torch.cuda.device(input.device):
        nbytes = lib.mrefsr_dcn_workspace_bytes(b, c, h, w, co, kh, kw, s[0], s[1], p[0], p[1], d[0], d[1], groups, dg,
                                                _default_mode, 1)
        ws, ws_bytes = _lib.workspace(nbytes, input.device)
        rc = lib.mrefsr_modulated_deform_conv_backward(
            _lib.ptr(input), _lib.ptr(weight), _lib.ptr(offset), _lib.ptr(mask), _lib.ptr(grad_output), _lib.ptr(gi),
            _lib.ptr(gw), _lib.ptr(gb), _lib.ptr(go), _lib.ptr(gm), b, c, h, w, co, kh, kw, s[0], s[1], p[0], p[1], d[0],
            d[1], groups, dg, int(with_bias), _default_mode, ws, ws_bytes, _lib.stream_ptr(input.device))
    _lib.check(rc, 'mrefsr_modulated_deform_conv_backward')
    return gi, go, gm, gw, gb


class DeformConvFunction(Function):
    """DCNv1 (basicsr/ops/dcn/deform_conv.py:33-118): the same kernels with an implicit all-ones mask and no bias.
    `im2col_step` is accepted for signature compatibility; the whole batch is one launch here."""

    @staticmethod
    def forward(ctx, input, offset, weight, stride=1, padding=0, dilation=1, groups=1, deformable_groups=1,
                im2col_step=64):
        if input is not None and input.dim() != 4:
            raise ValueError(f'Expected 4D tensor as input, got {input.dim()}D tensor instead.')
        ctx.stride, ctx.padding, ctx.dilation = _pair(stride), _pair(padding), _pair(dilation)
        ctx.groups = groups
        ctx.deformable_groups = deformable_groups
        ctx.im2col_step = im2col_step
        if not input.is_cuda:
            raise NotImplementedError
        _lib.require_cuda(offset, weight)
        cur = min(im2col_step, input.shape[0])
        assert (input.shape[0] % cur) == 0, 'im2col step must divide batchsize'
        kh, kw = weight.shape[2:4]
        ho, wo = _out_hw(input.shape[2], input.shape[3], kh, kw, ctx.stride, ctx.padding, ctx.dilation)
        if ho <= 0 or wo <= 0:
            raise ValueError('convolution input is too small (output would be %dx%d)' % (ho, wo))
        ctx.in_dtype = input.dtype
        x, off, wgt = (t.contiguous().float() for t in (input, offset, weight))
        ctx.save_for_backward(x, off, wgt)
        out = dcn_forward_raw(x, off, None, wgt, None, ctx.stride, ctx.padding, ctx.dilation, groups, deformable_groups)
        return out.to(input.dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        if not grad_output.is_cuda:
            raise NotImplementedError
        x, off, wgt = ctx.saved_tensors
        need_io = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        gi, go, _, gw, _ = dcn_backward_raw(x, off, None, wgt, grad_output.contiguous().float(), ctx.stride, ctx.padding,
                                            ctx.dilation, ctx.groups, ctx.deformable_groups, False, need_input=need_io,
                                            need_offset=need_io, need_weight=ctx.needs_input_grad[2])
        dt = ctx.in_dtype
        cast = (lambda t: None if t is None else t.to(dt))
        return (cast(gi), cast(go), cast(gw), None, None, None, None, None, None)


deform_conv = DeformConvFunction.apply


class DeformConv(nn.Module):
    """Same constructor, parameter (weight) and init as deform_conv.py:191-245."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deformable_groups=1, bias=False):
        super().__init__()
        assert not bias
        assert in_channels % groups == 0, f'in_channels {in_channels} is not divisible by groups {groups}'
        assert out_channels % groups == 0, f'out_channels {out_channels} is not divisible by groups {groups}'
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _pair(kernel_size)
        self.stride = _pair(stride)
        self.padding = _pair(padding)
        self.dilation = _pair(dilation)
        self.groups = groups
        self.deformable_groups = deformable_groups
        self.transposed = False
        self.output_padding = _single(0)
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels // self.groups, *self.kernel_size))
        self.reset_parameters()

    def reset_parameters(self):
        n = self.in_channels
        for k in self.kernel_size:
            n *= k
        stdv = 1. / math.sqrt(n)
        self.weight.data.uniform_(-stdv, stdv)

    def forward(self, x, offset):
        input_pad = (x.size(2) < self.kernel_size[0] or x.size(3) < self.kernel_size[1])
        if input_pad:
            pad_h = max(self.kernel_size[0] - x.size(2), 0)
            pad_w = max(self.kernel_size[1] - x.size(3), 0)
            x = torch.nn.functional.pad(x, (0, pad_w, 0, pad_h), 'constant', 0).contiguous()
            offset = torch.nn.functional.pad(offset, (0, pad_w, 0, pad_h), 'constant', 0).contiguous()
        out = deform_conv(x, offset, self.weight, self.stride, self.padding, self.dilation, self.groups,
                          self.deformable_groups)
        if input_pad:
            out = out[:, :, :out.size(2) - pad_h, :out.size(3) - pad_w].contiguous()
        return out


class DeformConvPack(DeformConv):
    """deform_conv.py:248-286: adds the zero-initialised conv_offset that predicts the offsets."""

    _version = 2

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.conv_offset = nn.Conv2d(self.in_channels,
                                     self.deformable_groups * 2 * self.kernel_size[0] * self.kernel_size[1],
                                     kernel_size=self.kernel_size, stride=_pair(self.stride),
                                     padding=_pair(self.padding), dilation=_pair(self.dilation), bias=True)
        self.init_offset()

    def init_offset(self):
        self.conv_offset.weight.data.zero_()
        self.conv_offset.bias.data.zero_()

    def forward(self, x):
        offset = self.conv_offset(x)
        return deform_conv(x, offset, self.weight, self.stride, self.padding, self.dilation, self.groups,
                           self.deformable_groups)


class ModulatedDeformConv(nn.Module):
    """Same constructor, parameters (weight, bias) and init as deform_conv.py:289-333."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deformable_groups=1, bias=True):
        super().__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _pair(kernel_size)
        self.stride = stride
        self.padding = padding
        self.dilation = dilation
        self.groups = groups
        self.deformable_groups = deformable_groups
        self.with_bias = bias
        self.transposed = False
        self.output_padding = _single(0)
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels // groups, *self.kernel_size))
        if bias:
            self.bias = nn.Parameter(torch.Tensor(out_channels))
        else:
            self.register_parameter('bias', None)
        self.init_weights()

    def init_weights(self):
        n = self.in_channels
        for k in self.kernel_size:
            n *= k
        stdv = 1. / math.sqrt(n)
        self.weight.data.uniform_(-stdv, stdv)
        if self.bias is not None:
            self.bias.data.zero_()

    def forward(self, x, offset, mask):
        return modulated_deform_conv(x, offset, mask, self.weight, self.bias, self.stride, self.padding, self.dilation,
                                     self.groups, self.deformable_groups)


class ModulatedDeformConvPack(ModulatedDeformConv):
    """deform_conv.py:336-379: adds the zero-initialised conv_offset that predicts offsets and masks."""

    _version = 2

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.conv_offset = nn.Conv2d(self.in_channels,
                                     self.deformable_groups * 3 * self.kernel_size[0] * self.kernel_size[1],
                                     kernel_size=self.kernel_size, stride=_pair(self.stride),
                                     padding=_pair(self.padding), dilation=_pair(self.dilation), bias=True)
        self.init_weights()

    def init_weights(self):
        super().init_weights()
        if hasattr(self, 'conv_offset'):
            self.conv_offset.weight.data.zero_()
            self.conv_offset.bias.data.zero_()

    def forward(self, x):
        out = self.conv_offset(x)
        o1, o2, mask = torch.chunk(out, 3, dim=1)
        offset = torch.cat((o1, o2), dim=1)
        mask = torch.sigmoid(mask)
        return modulated_deform_conv(x, offset, mask, self.weight, self.bias, self.stride, self.padding, self.dilation,
                                     self.groups, self.deformable_groups)


# ---------------------------------------------------------------------------------------------------
# the five functions the reference's pybind module exports (deform_conv_ext.cpp:150-164), same argument order,
# so that basicsr/ops/dcn/deform_conv.py can bind `deform_conv_ext = mrefsr_b200.dcn.ext` unchanged
# ---------------------------------------------------------------------------------------------------
class _Ext:
    @staticmethod
    def modulated_deform_conv_forward(input, weight, bias, ones, offset, mask, output, columns, kernel_h, kernel_w,
                                      stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
                                      deformable_group, with_bias):
        if not input.is_cuda:
            raise RuntimeError('modulated deform conv is not implemented on CPU')  # deform_conv_ext.cpp:124
        if not input.is_contiguous():
            raise RuntimeError('input tensor has to be contiguous')                # deform_conv_cuda.cpp:497
        if not weight.is_contiguous():
            raise RuntimeError('weight tensor has to be contiguous')
        if weight.shape[2] != kernel_h or weight.shape[3] != kernel_w:
            raise RuntimeError("Input shape and kernel shape won't match: (%d x %d vs %d x %d)." %
                               (kernel_h, kernel_w, weight.shape[2], weight.shape[3]))
        out = dcn_forward_raw(input.float(), offset.contiguous().float(), mask.contiguous().float(), weight.float(),
                              bias.contiguous().float() if with_bias else None, (stride_h, stride_w), (pad_h, pad_w),
                              (dilation_h, dilation_w), group, deformable_group)
        output.view(out.shape).copy_(out)

    @staticmethod
    def modulated_deform_conv_backward(input, weight, bias, ones, offset, mask, columns, grad_input, grad_weight,
                                       grad_bias, grad_offset, grad_mask, grad_output, kernel_h, kernel_w, stride_h,
                                       stride_w, pad_h, pad_w, dilation_h, dilation_w, group, deformable_group,
                                       with_bias):
        if not input.is_cuda:
            raise RuntimeError('modulated deform conv is not implemented on CPU')  # deform_conv_ext.cpp:146
        lib = _lib.lib()
        b, c, h, w = input.shape
        co = weight.shape[0]
        for t in (input, weight, offset, mask, grad_output, grad_input, grad_weight, grad_offset, grad_mask):
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise RuntimeError('deform_conv_ext shim: fp32 contiguous tensors only')
        with torch.cuda.device(input.device):
            nbytes = lib.mrefsr_dcn_workspace_bytes(b, c, h, w, co, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                                                    dilation_h, dilation_w, group, deformable_group, _default_mode, 1)
            ws, ws_bytes = _lib.workspace(nbytes, input.device)
            rc = lib.mrefsr_modulated_deform_conv_backward(
                _lib.ptr(input), _lib.ptr(weight), _lib.ptr(offset), _lib.ptr(mask), _lib.ptr(grad_output),
                _lib.ptr(grad_input), _lib.ptr(grad_weight), _lib.ptr(grad_bias) if with_bias else None,
                _lib.ptr(grad_offset), _lib.ptr(grad_mask), b, c, h, w, co, kernel_h, kernel_w, stride_h, stride_w,
                pad_h, pad_w, dilation_h, dilation_w, group, deformable_group, int(with_bias), _default_mode, ws,
                ws_bytes, _lib.stream_ptr(input.device))
        _lib.check(rc, 'mrefsr_modulated_deform_conv_backward')

    # DCNv1 exports (deform_conv_ext.cpp:52-105); note the reference's (W, H) argument order
    @staticmethod
    def deform_conv_forward(input, weight, offset, output, columns, ones, kW, kH, dW, dH, padW, padH, dilationW,
                            dilationH, group, deformable_group, im2col_step):
        if not input.is_cuda:
            raise RuntimeError('deform conv is not implemented on CPU')          # deform_conv_ext.cpp:63
        out = dcn_forward_raw(input.contiguous().float(), offset.contiguous().float(), None, weight.contiguous().float(),
                              None, (dH, dW), (padH, padW), (dilationH, dilationW), group, deformable_group)
        output.view(out.shape).copy_(out)
        return 1

    @staticmethod
    def deform_conv_backward_input(input, offset, gradOutput, gradInput, gradOffset, weight, columns, kW, kH, dW, dH,
                                   padW, padH, dilationW, dilationH, group, deformable_group, im2col_step):
        if not input.is_cuda:
            raise RuntimeError('deform conv is not implemented on CPU')
        gi, go, _, _, _ = dcn_backward_raw(input.contiguous().float(), offset.contiguous().float(), None,
                                           weight.contiguous().float(), gradOutput.contiguous().float(), (dH, dW),
                                           (padH, padW), (dilationH, dilationW), group, deformable_group, False,
                                           need_weight=False)
        gradInput.copy_(gi)
        gradOffset.copy_(go)
        return 1

    @staticmethod
    def deform_conv_backward_parameters(input, offset, gradOutput, gradWeight, columns, ones, kW, kH, dW, dH, padW,
                                        padH, dilationW, dilationH, group, deformable_group, scale, im2col_step):
        if not input.is_cuda:
            raise RuntimeError('deform conv is not implemented on CPU')
        kshape = (gradWeight.shape[0], input.shape[1] // group, kH, kW)
        wdummy = torch.empty(kshape, dtype=torch.float32, device=input.device)
        _, _, _, gw, _ = dcn_backward_raw(input.contiguous().float(), offset.contiguous().float(), None, wdummy,
                                          gradOutput.contiguous().float(), (dH, dW), (padH, padW),
                                          (dilationH, dilationW), group, deformable_group, False, need_input=False,
                                          need_offset=False)
        gradWeight.add_(gw.view_as(gradWeight), alpha=scale)        # accumulates, like the reference
        return 1


ext = _Ext()
