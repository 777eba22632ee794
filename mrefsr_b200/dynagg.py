"""DynAgg: DCNv2 whose offsets are initialised with the matcher's pre-offsets.

Drop-in for basicsr.archs.ref_mrapa_restoration_arch.DynAgg (:11-76): same constructor, same parameters
(weight, bias, conv_offset_mask.{weight,bias}), same forward(x, pre_offset).  The chunk / cat / repeat /
zeros_like / strided scatter / add / sigmoid sequence (:55-68) is one kernel, and the reference's host-syncing
``if offset_mean > 100`` check (:69-73, which also references an undefined ``logger``) is replaced by an
asynchronous device-side accumulator readable through ``last_offset_abs_mean()``.
``forward_fused(x, max_idx, flow_scale)`` takes the matcher's arg-max map instead of pre-offsets and builds offsets
and masks inside the DCN gather, in the forward and (DynAggFusedFunction) in the backward.
"""
import torch
from torch import nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib
from .mmcv_ops import ModulatedDeformConv2d, modulated_deform_conv2d


class DynAggOffsetsFunction(Function):
    """(conv_out [B,3*dg*K,H,W], pre_offset [B,K,H,W,2]) -> (offset [B,2*dg*K,H,W], mask [B,dg*K,H,W])."""

    @staticmethod
    def forward(ctx, conv_out, pre_offset, dg, stats):
        _lib.require_cuda(conv_out, pre_offset)
        ctx.in_dtype = conv_out.dtype
        from .trunk import to_nchw
        co = to_nchw(conv_out.float())
        pre = pre_offset.contiguous().float()
        b, ch, h, w = co.shape
        k = pre.shape[1]
        if ch != 3 * dg * k or tuple(pre.shape) != (b, k, h, w, 2):
            raise ValueError('expected conv_out [B,3*dg*K,H,W] and pre_offset [B,K,H,W,2]')
        offset = torch.empty(b, 2 * dg * k, h, w, dtype=torch.float32, device=co.device)
        mask = torch.empty(b, dg * k, h, w, dtype=torch.float32, device=co.device)
        with torch.cuda.device(co.device):
            rc = _lib.lib().mrefsr_dynagg_offsets(_lib.ptr(co), _lib.ptr(pre), _lib.ptr(offset), _lib.ptr(mask),
                                                  _lib.ptr(stats), b, dg, k, h, w, _lib.stream_ptr(co.device))
        _lib.check(rc, 'mrefsr_dynagg_offsets')
        ctx.save_for_backward(mask)
        return offset.to(conv_out.dtype), mask.to(conv_out.dtype)

    @staticmethod
    @once_differentiable
    def backward(ctx, g_offset, g_mask):
        (mask,) = ctx.saved_tensors
        # d offset / d conv_out = 1 on the first 2*dg*K channels; d sigmoid = m (1 - m) on the rest
        g = torch.cat((g_offset.float(), g_mask.float() * mask * (1 - mask)), dim=1)
        return g.to(ctx.in_dtype), None, None, None


class DynAggDCNFunction(Function):
    """Training path of DynAgg.forward as ONE autograd node: (x, conv_out, pre_offset, weight, bias) -> DCNv2 output.

    Same arithmetic as DynAggOffsetsFunction followed by ModulatedDeformConvFunction (the reference's operator
    boundaries, ref_mrapa_restoration_arch.py:55-76), but offsets / masks and their gradients stay fp32 tensors of this
    node instead of crossing two Function boundaries: under bf16 autocast that boundary costs eight cast passes over the
    216-plane tensor per call, and the glue backward (mul, mul, cat) is one kernel.  3x3 / stride 1 / padding 1 /
    dilation 1 / groups 1 only (what MRefSR uses); DynAgg.forward falls back to the two Functions otherwise."""

    @staticmethod
    def forward(ctx, x, conv_out, pre_offset, weight, bias, dg, stats, out_slope=1.0, out_like_conv=False):
        """out_slope != 1: a leaky ReLU on the output (the activation MRefSR applies after DynAgg,
        ref_mrapa_restoration_arch.py:229) as part of this node; out_like_conv: return the output in conv_out's dtype and
        layout (the trunk's) instead of x's -- both ride on the one conversion pass of the result."""
        from .dcn import dcn_forward_raw, _nchw
        _lib.require_cuda(x, conv_out, pre_offset, weight, bias)
        ctx.conv_dtype, ctx.x_dtype, ctx.dg = conv_out.dtype, x.dtype, dg
        ctx.conv_cl = conv_out.dim() == 4 and not conv_out.is_contiguous() and \
            conv_out.is_contiguous(memory_format=torch.channels_last)
        ctx.with_bias = bias is not None
        ctx.w_dtype = weight.dtype
        x32, co = _nchw(x), _nchw(conv_out)
        pre = pre_offset.contiguous().float()
        b, ch, h, w = co.shape
        k = pre.shape[1]
        if ch != 3 * dg * k or tuple(pre.shape) != (b, k, h, w, 2):
            raise ValueError('expected conv_out [B,3*dg*K,H,W] and pre_offset [B,K,H,W,2]')
        offset = torch.empty(b, 2 * dg * k, h, w, dtype=torch.float32, device=co.device)
        mask = torch.empty(b, dg * k, h, w, dtype=torch.float32, device=co.device)
        with torch.cuda.device(co.device):
            rc = _lib.lib().mrefsr_dynagg_offsets(_lib.ptr(co), _lib.ptr(pre), _lib.ptr(offset), _lib.ptr(mask),
                                                  _lib.ptr(stats), b, dg, k, h, w, _lib.stream_ptr(co.device))
        _lib.check(rc, 'mrefsr_dynagg_offsets')
        wgt = weight.contiguous().float()
        bs = bias.contiguous().float() if bias is not None else None
        out = dcn_forward_raw(x32, offset, mask, wgt, bs, (1, 1), (1, 1), (1, 1), 1, dg)
        ctx.out_slope = float(out_slope)
        from .trunk import from_nchw_f32
        if out_like_conv:
            res = from_nchw_f32(out, conv_out.dtype, ctx.conv_cl, slope=ctx.out_slope)
        else:
            if ctx.out_slope != 1.0:
                out = torch.nn.functional.leaky_relu_(out, ctx.out_slope)
            res = out.to(x.dtype)
        if ctx.out_slope != 1.0:
            ctx.save_for_backward(x32, offset, mask, wgt, res)
        else:
            ctx.save_for_backward(x32, offset, mask, wgt)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        from .dcn import dcn_backward_raw, _nchw
        from .trunk import to_nchw_f32
        if ctx.out_slope != 1.0:
            x32, offset, mask, wgt, res = ctx.saved_tensors
            if grad_output.dtype != res.dtype:
                grad_output = grad_output.to(res.dtype)
            g32 = to_nchw_f32(grad_output, gate=res, slope=ctx.out_slope)
        else:
            x32, offset, mask, wgt = ctx.saved_tensors
            g32 = _nchw(grad_output)
        need_conv = ctx.needs_input_grad[1]
        gi, go, gm, gw, gb = dcn_backward_raw(x32, offset, mask, wgt, g32, (1, 1), (1, 1), (1, 1), 1, ctx.dg,
                                              ctx.with_bias, need_input=ctx.needs_input_grad[0], need_offset=need_conv,
                                              need_weight=ctx.needs_input_grad[3])
        g_conv = None
        if need_conv:
            b, mc, h, w = mask.shape
            k = mc // ctx.dg
            g_conv = torch.empty(b, 3 * mc, h, w, dtype=torch.float32, device=mask.device)
            with torch.cuda.device(mask.device):
                rc = _lib.lib().mrefsr_dynagg_offsets_backward(_lib.ptr(go), _lib.ptr(gm), _lib.ptr(mask), _lib.ptr(g_conv), b,
                                                               ctx.dg, k, h, w, _lib.stream_ptr(mask.device))
            _lib.check(rc, 'mrefsr_dynagg_offsets_backward')
            if ctx.conv_cl or ctx.conv_dtype != torch.float32:
                from .trunk import from_nchw_f32
                g_conv = from_nchw_f32(g_conv, ctx.conv_dtype, ctx.conv_cl)
        cast = (lambda t, dt: None if t is None else t.to(dt))
        return (cast(gi, ctx.x_dtype), g_conv, None, cast(gw, ctx.w_dtype),
                gb if ctx.with_bias and ctx.needs_input_grad[4] else None, None, None, None, None)


class DynAggFusedFunction(Function):
    """Training path of DynAgg.forward_fused as ONE autograd node: (x, conv_out, max_idx, weight, bias) -> DCNv2 output.

    The forward is the launch `dcn.dynagg_dcn_forward` makes (offsets / masks assembled inside the gather from the raw
    conv_offset_mask output and the matcher's arg-max map); the backward reads the same source
    (mrefsr_dynagg_dcn_backward), so neither pass writes pre-offset, offset or mask tensors, and the gradient of
    conv_out comes straight out of the coordinate kernel.  out_slope / out_like_conv as in DynAggDCNFunction."""

    @staticmethod
    def forward(ctx, x, conv_out, max_idx, flow_scale, weight, bias, dg, out_slope=1.0, out_like_conv=False):
        from .dcn import dynagg_dcn_forward, _nchw
        from .trunk import from_nchw_f32, is_channels_last
        _lib.require_cuda(x, conv_out, max_idx, weight, bias)
        ctx.conv_dtype, ctx.x_dtype, ctx.w_dtype = conv_out.dtype, x.dtype, weight.dtype
        ctx.conv_cl = is_channels_last(conv_out)
        ctx.with_bias, ctx.dg, ctx.flow_scale = bias is not None, dg, int(flow_scale)
        x32 = x.float()
        if not is_channels_last(x32):
            x32 = x32.contiguous()
        co, wgt, mi = _nchw(conv_out), weight.contiguous().float(), max_idx.contiguous()
        out = dynagg_dcn_forward(x32, co, mi, flow_scale, wgt, bias, dg, out_channels_last=False)
        ctx.out_slope = float(out_slope)
        if out_like_conv:
            res = from_nchw_f32(out, conv_out.dtype, ctx.conv_cl, slope=ctx.out_slope)
        else:
            if ctx.out_slope != 1.0:
                out = torch.nn.functional.leaky_relu_(out, ctx.out_slope)
            res = out.to(x.dtype)
        if ctx.out_slope != 1.0:
            ctx.save_for_backward(x32, co, mi, wgt, res)
        else:
            ctx.save_for_backward(x32, co, mi, wgt)
        return res

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        from .dcn import dynagg_dcn_backward_raw, _nchw
        from .trunk import from_nchw_f32, to_nchw_f32
        if ctx.out_slope != 1.0:
            x32, co, mi, wgt, res = ctx.saved_tensors
            if grad_output.dtype != res.dtype:
                grad_output = grad_output.to(res.dtype)
            g32 = to_nchw_f32(grad_output, gate=res, slope=ctx.out_slope)
        else:
            x32, co, mi, wgt = ctx.saved_tensors
            g32 = _nchw(grad_output)
        gi, g_conv, gw, gb = dynagg_dcn_backward_raw(x32, co, mi, ctx.flow_scale, wgt, g32, ctx.dg, ctx.with_bias,
                                                     need_input=ctx.needs_input_grad[0],
                                                     need_conv=ctx.needs_input_grad[1],
                                                     need_weight=ctx.needs_input_grad[4])
        if g_conv is not None and (ctx.conv_cl or ctx.conv_dtype != torch.float32):
            g_conv = from_nchw_f32(g_conv, ctx.conv_dtype, ctx.conv_cl)
        cast = (lambda t, dt: None if t is None else t.to(dt))
        return (cast(gi, ctx.x_dtype), g_conv, None, None, cast(gw, ctx.w_dtype),
                gb if ctx.with_bias and ctx.needs_input_grad[5] else None, None, None, None)


class DynAgg(ModulatedDeformConv2d):

    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation=1, groups=1,
                 deform_groups=1, extra_offset_mask=True):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, deform_groups)
        self.extra_offset_mask = extra_offset_mask
        channels_ = self.deform_groups * 3 * self.kernel_size[0] * self.kernel_size[1]
        self.conv_offset_mask = nn.Conv2d(self.in_channels, channels_, kernel_size=self.kernel_size,
                                          stride=self.stride, padding=self.padding, bias=True)
        self.init_offset()
        self.fused_autograd = True       # forward(): one autograd node (DynAggDCNFunction) instead of the two operator Functions
        self._stats = None
        self._stats_count = 0

    def init_offset(self):
        self.conv_offset_mask.weight.data.zero_()
        self.conv_offset_mask.bias.data.zero_()

    def last_offset_abs_mean(self):
        """mean |learned offset| of the last forward (one device->host read, only when asked)."""
        if self._stats is None or self._stats_count == 0:
            return None
        return float(self._stats.item()) / self._stats_count

    def forward_fused(self, x, max_idx, flow_scale, out_slope=1.0, out_like_conv=False):
        """Same result as forward(x, pre_offset) where pre_offset is the matcher's shifted flow at this scale
        (max_idx int64 [B, H/flow_scale - 2, W/flow_scale - 2]), but offsets / masks / pre-offsets never touch HBM.
        With grad enabled and x or a parameter requiring grad this is one autograd node (DynAggFusedFunction) whose
        backward reads the same source; otherwise the inference path.  out_slope: leaky ReLU applied to the result;
        out_like_conv: the result in the dtype / layout of the offset convolution's output (the trunk's)."""
        from .dcn import dynagg_dcn_forward
        from . import trunk as T
        if not (tuple(self.kernel_size) == (3, 3) and tuple(self.stride) == (1, 1) and tuple(self.padding) == (1, 1)
                and tuple(self.dilation) == (1, 1) and self.groups == 1):
            raise NotImplementedError('forward_fused serves the configuration MRefSR uses (3x3, stride 1, padding 1, '
                                      'dilation 1, groups 1: ref_mrapa_restoration_arch.py:146-158); use forward() with '
                                      'materialised pre-offsets for anything else')
        feat = x[1] if self.extra_offset_mask else x
        if self.extra_offset_mask:
            x = x[0]
        if torch.is_grad_enabled() and (x.requires_grad or feat.requires_grad or
                                        any(p.requires_grad for p in self.parameters())):
            out = T.conv_act(feat, self.conv_offset_mask)       # (training: bias add and its gradient fused)
            return DynAggFusedFunction.apply(x, out, max_idx, flow_scale, self.weight, self.bias, self.deform_groups,
                                             out_slope, out_like_conv)
        if T.fast_ok(feat):    # the DCN reads planes: bias (+ the NHWC -> NCHW conversion of a channels-last conv) in one pass
            out = T.conv_bias_to_nchw(feat, self.conv_offset_mask)
        else:
            out = self.conv_offset_mask(feat)
        y = dynagg_dcn_forward(x, out, max_idx, flow_scale, self.weight, self.bias, self.deform_groups,
                               out_slope=out_slope)
        if out_like_conv:      # (the convolution keeps its input's layout; conv_bias_to_nchw hands back planes)
            y = y.to(dtype=out.dtype, memory_format=torch.channels_last if T.is_channels_last(feat) else
                     torch.contiguous_format)
        return y

    def forward(self, x, pre_offset, out_slope=1.0, out_like_conv=False):
        """Reference signature forward(x, pre_offset).  out_slope / out_like_conv (fused autograd node only): apply the
        leaky ReLU that follows DynAgg in MRefSR and return the result in the offset convolution's dtype / layout."""
        from . import trunk as T
        if self.extra_offset_mask:
            out = T.conv_act(x[1], self.conv_offset_mask)       # (training: bias add and its gradient fused)
            x = x[0]
        else:
            out = T.conv_act(x, self.conv_offset_mask)
        if self._stats is None or self._stats.device != out.device:
            self._stats = torch.zeros(1, dtype=torch.float32, device=out.device)
        self._stats.zero_()
        if self.fused_autograd and (tuple(self.kernel_size) == (3, 3) and tuple(self.stride) == (1, 1) and
                                    tuple(self.padding) == (1, 1) and tuple(self.dilation) == (1, 1) and self.groups == 1):
            self._stats_count = out.numel() // 3 * 2
            return DynAggDCNFunction.apply(x, out, pre_offset, self.weight, self.bias, self.deform_groups, self._stats,
                                           out_slope, out_like_conv)
        if out_slope != 1.0 or out_like_conv:
            raise NotImplementedError('out_slope / out_like_conv need the fused autograd node (3x3, stride 1, padding 1)')
        offset, mask = DynAggOffsetsFunction.apply(out, pre_offset, self.deform_groups, self._stats)
        self._stats_count = offset.numel()
        return modulated_deform_conv2d(x, offset, mask, self.weight, self.bias, self.stride, self.padding,
                                       self.dilation, self.groups, self.deform_groups)
