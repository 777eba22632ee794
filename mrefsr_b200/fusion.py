"""Multi-reference attention fusion: host-side mirror of MRAPAFusion
(basicsr/archs/ref_mrapa_restoration_arch.py:262-348) with the attention core (:321-335) on csrc/fusion.cu.

``MRAPAFusion`` keeps the reference's constructor, parameter names (state-dict keys conv_emb1.0.*,
conv_emb1.1.weight, conv_emb2.*, conv_ass.*, feat_fusion.*, spatial_attn*.*) and forward signature
``forward(target, refs: list[Tensor])``; the plain convolutions stay cuDNN library calls.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib
from . import trunk as T


class MRAPAAttentionFunction(Function):
    """out[n,Cv,h,w] = sum_t softmax_t(<emb_t[n,:,y,x], emb[n,t,:,y,x]>) * ass[n,t,:,y,x]."""

    @staticmethod
    def forward(ctx, emb_t, emb, ass, t):
        _lib.require_cuda(emb_t, emb, ass)
        ctx.in_dtype = emb_t.dtype
        ctx.in_cl = tuple(T.is_channels_last(x) for x in (emb_t, emb, ass))
        q, k, v = (T.to_nchw_f32(x) for x in (emb_t, emb, ass))
        n, c, h, w = q.shape
        if k.shape[0] != n * t or k.shape[1] != c or v.shape[0] != n * t or k.shape[2:] != q.shape[2:] \
                or v.shape[2:] != q.shape[2:]:
            raise ValueError('expected emb_t [n,C,h,w], emb [n*t,C,h,w], ass [n*t,Cv,h,w]')
        cv = v.shape[1]
        out = torch.empty(n, cv, h, w, dtype=torch.float32, device=q.device)
        need = any(ctx.needs_input_grad[:3])
        prob = torch.empty(n, t, h, w, dtype=torch.float32, device=q.device) if need else None
        with torch.cuda.device(q.device):
            rc = _lib.lib().mrefsr_mrapa_attention_forward(_lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(out),
                                                           _lib.ptr(prob), n, t, c, cv, h, w,
                                                           _lib.stream_ptr(q.device))
        _lib.check(rc, 'mrefsr_mrapa_attention_forward')
        if need:
            ctx.save_for_backward(q, k, v, prob)
        ctx.t = t
        return T.from_nchw_f32(out, emb_t.dtype, ctx.in_cl[0])

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        q, k, v, prob = ctx.saved_tensors
        go = T.to_nchw_f32(grad_out)
        n, c, h, w = q.shape
        cv = v.shape[1]
        gq, gk, gv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        with torch.cuda.device(q.device):
            rc = _lib.lib().mrefsr_mrapa_attention_backward(_lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(prob),
                                                            _lib.ptr(go), _lib.ptr(gq), _lib.ptr(gk), _lib.ptr(gv), n,
                                                            ctx.t, c, cv, h, w, _lib.stream_ptr(q.device))
        _lib.check(rc, 'mrefsr_mrapa_attention_backward')
        dt = ctx.in_dtype      # gradients go back in the dtype AND layout the inputs came in (bf16 channels-last: one pass)
        return (T.from_nchw_f32(gq, dt, ctx.in_cl[0]), T.from_nchw_f32(gk, dt, ctx.in_cl[1]),
                T.from_nchw_f32(gv, dt, ctx.in_cl[2]), None)


def mrapa_attention(emb_t, emb, ass, t):
    """emb_t [n,C,h,w] (already scaled by C**-0.5), emb [n*t,C,h,w], ass [n*t,Cv,h,w] -> [n,Cv,h,w].
    Three bf16 tensors that need no gradient take the bf16-I/O kernel (`mrapa_attention_bf16`) when it serves them;
    the calls it refuses (more than 8 references, h*w % 4 != 0, planes not 8-byte aligned) run in fp32 and return bf16."""
    if (emb_t.dtype == emb.dtype == ass.dtype == torch.bfloat16 and
            not (torch.is_grad_enabled() and (emb_t.requires_grad or emb.requires_grad or ass.requires_grad)) and
            _bf16_kernel_serves(emb_t, emb, ass, t)):
        return mrapa_attention_bf16(emb_t, emb, ass, t)
    return MRAPAAttentionFunction.apply(emb_t, emb, ass, t)


def _bf16_kernel_serves(emb_t, emb, ass, t):
    """What mrefsr_mrapa_attention_forward_bf16 accepts: t <= 8, h*w % 4 == 0 and 8-byte-aligned tensors.  A tensor
    that is not contiguous is copied by mrapa_attention_bf16 into a fresh (aligned) allocation."""
    return (t <= 8 and emb_t.dim() == 4 and emb_t.shape[2] * emb_t.shape[3] % 4 == 0 and
            all(not x.is_contiguous() or x.data_ptr() % 8 == 0 for x in (emb_t, emb, ass)))


def mrapa_attention_bf16(emb_t, emb, ass, t):
    """bf16 tensors in, bf16 tensor out (inference): the fusion core is HBM-bound, so halving the bytes halves its time.
    Logits, softmax over the references and the weighted sum are computed in fp32; the result is rounded to nearest
    even.  Stated tolerance: 4e-3 of the output scale against the fp64 oracle on the same bf16-rounded inputs
    (tests/test_fusion_gpu.py::test_bf16_io)."""
    _lib.require_cuda(emb_t, emb, ass)
    n, c, h, w = emb_t.shape
    cv = ass.shape[1]
    if not all(x.dtype == torch.bfloat16 for x in (emb_t, emb, ass)):
        raise ValueError('mrapa_attention_bf16: bf16 tensors expected')
    if tuple(emb.shape) != (n * t, c, h, w) or tuple(ass.shape) != (n * t, cv, h, w):
        raise ValueError('expected emb_t [n,C,h,w], emb [n*t,C,h,w], ass [n*t,Cv,h,w]')
    q, k, v = emb_t.contiguous(), emb.contiguous(), ass.contiguous()
    out = torch.empty(n, cv, h, w, dtype=torch.bfloat16, device=q.device)
    with torch.cuda.device(q.device):
        rc = _lib.lib().mrefsr_mrapa_attention_forward_bf16(_lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(out), n, t, c, cv,
                                                            h, w, _lib.stream_ptr(q.device))
    _lib.check(rc, 'mrefsr_mrapa_attention_forward_bf16')
    return out


def mrapa_attention_nhwc(q_raw, k_raw, v_raw, t, bias_q=None, bias_k=None, bias_v=None, slope_q=None, slope_k=None,
                         q_scale=1.0):
    """Channels-last inference variant: inputs are the raw (bias-free) outputs of conv_emb1 / conv_emb2 / conv_ass as
    torch.channels_last tensors; bias, PReLU and the C^-0.5 scale are applied inside the kernel.
    q_raw [n,C,h,w], k_raw [n*t,C,h,w], v_raw [n*t,2C,h,w] -> channels_last [n,2C,h,w]."""
    _lib.require_cuda(q_raw, k_raw, v_raw)
    n, c, h, w = q_raw.shape
    cv = v_raw.shape[1]
    cl = torch.channels_last
    if not all(x.dtype == torch.float32 and x.is_contiguous(memory_format=cl) for x in (q_raw, k_raw, v_raw)):
        raise ValueError('expected fp32 torch.channels_last tensors')
    if tuple(k_raw.shape) != (n * t, c, h, w) or tuple(v_raw.shape) != (n * t, cv, h, w):
        raise ValueError('expected q_raw [n,C,h,w], k_raw [n*t,C,h,w], v_raw [n*t,Cv,h,w]')
    out = torch.empty(n, cv, h, w, dtype=torch.float32, device=q_raw.device, memory_format=cl)
    with torch.cuda.device(q_raw.device):
        rc = _lib.lib().mrefsr_mrapa_attention_nhwc(
            _lib.ptr(q_raw), _lib.ptr(k_raw), _lib.ptr(v_raw), _lib.ptr(bias_q), _lib.ptr(bias_k), _lib.ptr(bias_v),
            _lib.ptr(slope_q), 0 if slope_q is None else slope_q.numel(), _lib.ptr(slope_k),
            0 if slope_k is None else slope_k.numel(), float(q_scale), _lib.ptr(out), n, t, c, cv, h, w,
            _lib.stream_ptr(q_raw.device))
    _lib.check(rc, 'mrefsr_mrapa_attention_nhwc')
    return out


class MRAPAFusion(nn.Module):
    """Drop-in for basicsr.archs.ref_mrapa_restoration_arch.MRAPAFusion (same parameters and forward)."""

    def __init__(self, nf=64, ref_nf=256):
        super().__init__()
        self.patch_size = 3
        channels = ref_nf
        self.conv_emb1 = nn.Sequential(nn.Conv2d(nf, channels, 1), nn.PReLU())
        self.conv_emb2 = nn.Sequential(nn.Conv2d(ref_nf, channels, self.patch_size, 1, self.patch_size // 2),
                                       nn.PReLU())
        self.conv_ass = nn.Conv2d(ref_nf, channels * 2, self.patch_size, 1, self.patch_size // 2)
        self.scale = channels ** -0.5
        self.feat_fusion = nn.Conv2d(nf + channels * 2, nf, 1)
        self.spatial_attn = nn.Conv2d(nf + channels * 2, channels * 2, 1)
        self.spatial_attn_mul1 = nn.Conv2d(channels * 2, channels * 2, 3, padding=1)
        self.spatial_attn_mul2 = nn.Conv2d(channels * 2, channels * 2, 3, padding=1)
        self.spatial_attn_add1 = nn.Conv2d(channels * 2, channels * 2, 3, padding=1)
        self.spatial_attn_add2 = nn.Conv2d(channels * 2, channels * 2, 3, padding=1)
        self.lrelu = nn.LeakyReLU(negative_slope=0.1, inplace=True)

    def spatial_padding(self, feats):
        _, _, h, w = feats.size()
        pad_h = (4 - h % 4) % 4
        pad_w = (4 - w % 4) % 4
        if pad_h == 0 and pad_w == 0:      # F.pad would still copy the tensor
            return feats
        return F.pad(feats, [0, pad_w, 0, pad_h], mode='reflect')

    def forward(self, target, refs):
        return self.forward_stacked(target, torch.stack(refs, dim=1).flatten(0, 1), len(refs))

    def forward_stacked(self, target, refs, t):
        """Same as forward() with the t references already stacked: refs [n*t, ref_nf, h, w] (pairs laid out [n, t])."""
        n, _, h_input, w_input = target.size()
        target = self.spatial_padding(target)
        refs = self.spatial_padding(refs)
        if T.fast_ok(target, refs):
            return self._forward_fused_glue(target, refs, t, h_input, w_input)
        # multi-ref attention: one fused kernel instead of 3 permute copies + 2 batched matmuls (:321-335)
        # (autograd path; T.conv_act = conv -> [bias, lrelu] with the fused training epilogue where it applies)
        emb_t = self.conv_emb1(target) * self.scale
        emb = self.conv_emb2(refs)
        ass = T.conv_act(refs, self.conv_ass)
        refs = mrapa_attention(emb_t, emb, ass, t)
        if T.layout_of(target) == 1 and T.layout_of(refs) != 1:      # keep a channels-last trunk channels-last
            refs = refs.contiguous(memory_format=torch.channels_last)
        # spatial attention (:338-344)
        attn = T.conv_act(torch.cat([target, refs.to(target.dtype)], dim=1), self.spatial_attn, T.ACT_LEAKY, 0.1)
        attn_mul = T.conv_act(T.conv_act(attn, self.spatial_attn_mul1, T.ACT_LEAKY, 0.1), self.spatial_attn_mul2)
        attn_add = T.conv_act(T.conv_act(attn, self.spatial_attn_add1, T.ACT_LEAKY, 0.1), self.spatial_attn_add2)
        attn_mul = torch.sigmoid(attn_mul)
        refs = refs * attn_mul * 2 + attn_add
        feat = T.conv_act(torch.cat([target, refs.to(target.dtype)], dim=1), self.feat_fusion, T.ACT_LEAKY, 0.1)
        return feat[:, :, :h_input, :w_input]

    def _forward_fused_glue(self, target, refs, t, h_input, w_input):
        """Inference path: same arithmetic, every conv's bias / activation / scale epilogue in one pass and the
        spatial-attention modulation (sigmoid, * 2, + add, both conv biases) in one kernel."""
        c = self.conv_emb2[0].out_channels
        if T.layout_of(target) == 1 and T.layout_of(refs) == 1 and c in (64, 128, 256) and t <= 8:
            # channels-last: the attention kernel reads the raw convolution outputs and applies their bias / PReLU /
            # scale itself -- no epilogue pass over emb_t / emb / ass and no layout conversion
            cl = torch.channels_last
            q, k, v = (T.conv_raw(target, self.conv_emb1[0]).contiguous(memory_format=cl),
                       T.conv_raw(refs, self.conv_emb2[0]).contiguous(memory_format=cl),
                       T.conv_raw(refs, self.conv_ass).contiguous(memory_format=cl))
            refs = mrapa_attention_nhwc(q, k, v, t, self.conv_emb1[0].bias, self.conv_emb2[0].bias,
                                        self.conv_ass.bias, self.conv_emb1[1].weight, self.conv_emb2[1].weight,
                                        self.scale)
        else:
            emb_t = T.conv_bias_act(target, self.conv_emb1[0], prelu=self.conv_emb1[1], scale=self.scale)
            emb = T.conv_bias_act(refs, self.conv_emb2[0], prelu=self.conv_emb2[1])
            ass = T.conv_bias_act(refs, self.conv_ass)
            refs = mrapa_attention(emb_t, emb, ass, t)
            if T.layout_of(target) == 1:      # keep the channels-last trunk channels-last
                refs = T.to_nhwc(refs)
        attn = T.conv_bias_act(torch.cat([target, refs], dim=1), self.spatial_attn, T.ACT_LEAKY, 0.1)
        attn_mul = T.conv_raw(T.conv_bias_act(attn, self.spatial_attn_mul1, T.ACT_LEAKY, 0.1), self.spatial_attn_mul2)
        attn_add = T.conv_raw(T.conv_bias_act(attn, self.spatial_attn_add1, T.ACT_LEAKY, 0.1), self.spatial_attn_add2)
        refs = T.attn_modulate_(refs, T.dense(attn_mul), T.dense(attn_add), self.spatial_attn_mul2.bias,
                                self.spatial_attn_add2.bias)
        feat = T.conv_bias_act(torch.cat([target, refs], dim=1), self.feat_fusion, T.ACT_LEAKY, 0.1)
        return feat[:, :, :h_input, :w_input]
