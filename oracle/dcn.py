"""Oracle for DCNv2 (modulated deformable convolution) and the DynAgg glue.

TEST INFRASTRUCTURE, see oracle/__init__.py.

Restates
  * the sampling rule  basicsr/ops/dcn/src/deform_conv_cuda_kernel.cu:468-497 (bilinear, corners
    outside the image contribute 0) and :571-633 (im2col: h_im = h_out*stride - pad + i*dil + dy,
    value 0 unless -1 < h_im < H and -1 < w_im < W, times mask; offset channel 2*(g*K+k) is dy,
    +1 is dx; mask channel g*K+k),
  * the host side      basicsr/ops/dcn/src/deform_conv_cuda.cpp:490-569 (per-group
    out = W[g] . columns[g] + bias),
  * the backward       deform_conv_cuda.cpp:571-685 with kernels .cu:635-767; here the gradients
    are obtained by differentiating the restated forward (floor() has zero derivative, so the
    one-sided bilinear derivative of dmcn_get_coordinate_weight .cu:526-568 and the scatter
    weights of dmcn_get_gradient_weight .cu:499-524 are what autograd produces),
  * DynAgg.forward     basicsr/archs/ref_mrapa_restoration_arch.py:45-76 (offset/mask assembly).

Two implementations: a vectorised torch one (this file; fp32 or fp64) and a plain-C one
(dcn_ref.c, explicit loops, built by oracle/build.py) used as a second opinion and as the
multi-threaded CPU baseline.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))


def _pair(v):
    return (v, v) if isinstance(v, int) else tuple(v)


def sampling_positions(offset, kh, kw, stride, padding, dilation, dg, dtype, fp32_positions=False):
    """Sampling positions (him, wim), each [B, dg, kh*kw, Ho, Wo], of offset [B, 2*dg*kh*kw, Ho, Wo]:
    h_out*stride - pad + i*dil + offset (dy in channel 2*(g*K+k), dx in channel 2*(g*K+k)+1), in `dtype`.

    fp32_positions: the positions take the value of the fp32 sum (h_out*stride - pad + i*dil) + offset, one rounding,
    as the reference computes them (deform_conv_cuda_kernel.cu, modulated_deformable_im2col_gpu_kernel and
    modulated_deformable_col2im_coord_gpu_kernel: `h_in + i * dilation_h + offset_h` in scalar_t) and as the kernels
    of this package do.  Their derivative with respect to the offset stays 1 (straight-through).  The exact sum (the
    default) differs where that rounding carries a point across an integer, and the offset gradient jumps there."""
    sh, sw = stride
    ph, pw = padding
    dh, dw = dilation
    kk = kh * kw
    b, _, ho, wo = offset.shape
    off = offset.view(b, dg, kk, 2, ho, wo)
    ys = (torch.arange(ho, dtype=dtype) * sh - ph).view(1, 1, 1, ho, 1)
    xs = (torch.arange(wo, dtype=dtype) * sw - pw).view(1, 1, 1, 1, wo)
    ki = (torch.arange(kk) // kw).to(dtype).view(1, 1, kk, 1, 1) * dh
    kj = (torch.arange(kk) % kw).to(dtype).view(1, 1, kk, 1, 1) * dw
    him = ys + ki + off[:, :, :, 0]
    wim = xs + kj + off[:, :, :, 1]
    if fp32_positions:
        # |fp32 sum - exact sum| is one rounding of the sum, so the difference and the re-addition are exact in fp64
        him = him + ((ys + ki).float() + off[:, :, :, 0].float() - him).detach()
        wim = wim + ((xs + kj).float() + off[:, :, :, 1].float() - wim).detach()
    return him, wim


def _columns(x, offset, mask, kh, kw, stride, padding, dilation, dg, fp32_positions=False):
    """Deformable im2col: [B, Cin, kh*kw, Ho*Wo] (value * mask).  fp32_positions: see sampling_positions."""
    b, cin, h, w = x.shape
    kk = kh * kw
    cg = cin // dg
    dt = x.dtype
    ho, wo = offset.shape[2:]
    msk = mask.view(b, dg, kk, ho, wo)
    him, wim = sampling_positions(offset, kh, kw, stride, padding, dilation, dg, dt, fp32_positions)
    inside = (him > -1) & (wim > -1) & (him < h) & (wim < w)
    hl = torch.floor(him)
    wl = torch.floor(wim)
    lh = him - hl
    lw = wim - wl
    hl = hl.long()
    wl = wl.long()
    xg = x.view(b, dg, cg, h * w)
    val = torch.zeros(b, dg, cg, kk, ho, wo, dtype=dt)
    for (dy, dx, wgt) in ((0, 0, (1 - lh) * (1 - lw)), (0, 1, (1 - lh) * lw),
                          (1, 0, lh * (1 - lw)), (1, 1, lh * lw)):
        yy = hl + dy
        xx = wl + dx
        ok = inside & (yy >= 0) & (yy <= h - 1) & (xx >= 0) & (xx <= w - 1)
        lin = (yy.clamp(0, h - 1) * w + xx.clamp(0, w - 1)).view(b, dg, 1, kk * ho * wo)
        g = torch.gather(xg, 3, lin.expand(b, dg, cg, kk * ho * wo)).view(b, dg, cg, kk, ho, wo)
        val = val + g * (wgt * ok.to(dt)).unsqueeze(2)
    val = val * msk.unsqueeze(2)
    return val.reshape(b, cin, kk, ho * wo), ho, wo


def modulated_deform_conv_oracle(x, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1,
                                 groups=1, deformable_groups=1, dtype=None, fp32_positions=False):
    """out[B, Cout, Ho, Wo]; argument meaning as ModulatedDeformConvFunction.forward
    (basicsr/ops/dcn/deform_conv.py:124-153).  fp32_positions: see sampling_positions."""
    dtype = dtype or x.dtype
    x, offset, mask, weight = (t.to(dtype) for t in (x, offset, mask, weight))
    stride, padding, dilation = _pair(stride), _pair(padding), _pair(dilation)
    cout, cin_g, kh, kw = weight.shape
    b = x.shape[0]
    cols, ho, wo = _columns(x, offset, mask, kh, kw, stride, padding, dilation, deformable_groups, fp32_positions)
    cols = cols.reshape(b, groups, cin_g * kh * kw, ho * wo)
    wmat = weight.reshape(groups, cout // groups, cin_g * kh * kw)
    out = torch.einsum('gok,bgkp->bgop', wmat, cols).reshape(b, cout, ho, wo)
    if bias is not None:
        out = out + bias.to(dtype).view(1, cout, 1, 1)
    return out


def modulated_deform_conv_backward_oracle(x, offset, mask, weight, bias, grad_output, stride=1, padding=0,
                                          dilation=1, groups=1, deformable_groups=1, dtype=None, fp32_positions=False):
    """(grad_input, grad_offset, grad_mask, grad_weight, grad_bias) as returned by
    ModulatedDeformConvFunction.backward (deform_conv.py:155-174).  fp32_positions: see sampling_positions."""
    dtype = dtype or x.dtype
    leaves = [t.detach().to(dtype).clone().requires_grad_(True) for t in (x, offset, mask, weight)]
    bl = None if bias is None else bias.detach().to(dtype).clone().requires_grad_(True)
    out = modulated_deform_conv_oracle(leaves[0], leaves[1], leaves[2], leaves[3], bl, stride, padding,
                                       dilation, groups, deformable_groups, dtype, fp32_positions)
    ins = leaves + ([bl] if bl is not None else [])
    grads = torch.autograd.grad(out, ins, grad_output.to(dtype), allow_unused=True)
    grads = [g if g is not None else torch.zeros_like(t) for g, t in zip(grads, ins)]
    return tuple(grads) + ((None,) if bl is None else ())


def dynagg_offsets_oracle(conv_out, pre_offset, deform_groups):
    """DynAgg glue (ref_mrapa_restoration_arch.py:55-68): raw conv_offset_mask output
    [B, 3*dg*9, H, W] + pre_offset [B, 9, H, W, 2] (x, y) -> (offset [B, 2*dg*9, H, W], mask)."""
    o1, o2, m = torch.chunk(conv_out, 3, dim=1)
    offset = torch.cat((o1, o2), dim=1).clone()
    pre = pre_offset.repeat(1, deform_groups, 1, 1, 1)
    offset[:, 0::2] += pre[..., 1]
    offset[:, 1::2] += pre[..., 0]
    return offset, torch.sigmoid(m)


# --------------------------------------------------------------------------------------
# plain-C second opinion / multi-threaded CPU baseline (oracle/dcn_ref.c)
# --------------------------------------------------------------------------------------
_clib = None


def c_lib():
    global _clib
    if _clib is None:
        path = os.path.join(_HERE, 'libdcn_ref.so')
        if not os.path.exists(path):
            from . import build
            build.build_c()
        _clib = ctypes.CDLL(path)
        fp = ctypes.POINTER(ctypes.c_float)
        _clib.dcn_ref_forward.argtypes = [fp, fp, fp, fp, fp, fp] + [ctypes.c_int] * 16
        _clib.dcn_ref_forward.restype = None
        _clib.dcn_ref_backward.argtypes = [fp] * 11 + [ctypes.c_int] * 16
        _clib.dcn_ref_backward.restype = None
    return _clib


def _fptr(t):
    return ctypes.cast(t.data_ptr(), ctypes.POINTER(ctypes.c_float)) if t is not None else None


def modulated_deform_conv_c(x, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1,
                            groups=1, deformable_groups=1):
    lib = c_lib()
    stride, padding, dilation = _pair(stride), _pair(padding), _pair(dilation)
    x, offset, mask, weight = (t.contiguous().float() for t in (x, offset, mask, weight))
    b, cin, h, w = x.shape
    cout, _, kh, kw = weight.shape
    ho = (h + 2 * padding[0] - (dilation[0] * (kh - 1) + 1)) // stride[0] + 1
    wo = (w + 2 * padding[1] - (dilation[1] * (kw - 1) + 1)) // stride[1] + 1
    out = torch.empty(b, cout, ho, wo)
    bb = bias.contiguous().float() if bias is not None else None
    lib.dcn_ref_forward(_fptr(x), _fptr(offset), _fptr(mask), _fptr(weight), _fptr(bb), _fptr(out),
                        b, cin, h, w, cout, kh, kw, stride[0], stride[1], padding[0], padding[1],
                        dilation[0], dilation[1], groups, deformable_groups, 1 if bb is not None else 0)
    return out


def modulated_deform_conv_backward_c(x, offset, mask, weight, bias, grad_output, stride=1, padding=0,
                                     dilation=1, groups=1, deformable_groups=1):
    lib = c_lib()
    stride, padding, dilation = _pair(stride), _pair(padding), _pair(dilation)
    x, offset, mask, weight, go = (t.contiguous().float() for t in (x, offset, mask, weight, grad_output))
    b, cin, h, w = x.shape
    cout, _, kh, kw = weight.shape
    gi, goff, gm, gw = (torch.zeros_like(t) for t in (x, offset, mask, weight))
    gb = torch.zeros(cout)
    lib.dcn_ref_backward(_fptr(x), _fptr(offset), _fptr(mask), _fptr(weight), _fptr(go),
                         _fptr(gi), _fptr(goff), _fptr(gm), _fptr(gw), _fptr(gb), None,
                         b, cin, h, w, cout, kh, kw, stride[0], stride[1], padding[0], padding[1],
                         dilation[0], dilation[1], groups, deformable_groups, 1 if bias is not None else 0)
    return gi, goff, gm, gw, (gb if bias is not None else None)
