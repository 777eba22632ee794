"""Parity of the CUDA DCNv2 (through the C ABI and the torch extension module) against the oracle, the golden vectors
generated from the reference's DynAgg, and -- when oracle/_ref holds the reference's own CUDA extension -- the
reference kernels."""
import os

import pytest
import torch

import mrefsr_b200 as M
import oracle
from mrefsr_b200 import dcn as D
from tests.util import rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 1e-3   # north star: DCN outputs within 1e-3 relative error in fp32


def _rand_problem(b, c, h, w, co, dg, seed, off_scale=2.0, groups=1, k=3, stride=1, pad=1, dil=1):
    g = torch.Generator().manual_seed(seed)
    ho = (h + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    wo = (w + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    x = torch.randn(b, c, h, w, generator=g)
    off = torch.randn(b, 2 * dg * k * k, ho, wo, generator=g) * off_scale
    mask = torch.rand(b, dg * k * k, ho, wo, generator=g)
    wgt = torch.randn(co, c // groups, k, k, generator=g) * (1.0 / (c * k * k) ** 0.5)
    bias = torch.randn(co, generator=g) * 0.1
    return x, off, mask, wgt, bias


@pytest.mark.parametrize('case', ['small', 'big_offsets'])
@pytest.mark.parametrize('mode', ['fp32', 'auto'])
def test_golden_forward_backward(golden, case, mode):
    g = golden('dynagg')
    dg = int(g(f'{case}.dg'))
    D.set_default_mode(mode)
    try:
        ts = [g(f'{case}.{k}').to(DEV).requires_grad_(True) for k in ('x', 'offset', 'mask', 'weight', 'bias')]
        y = M.modulated_deform_conv(ts[0], ts[1], ts[2], ts[3], ts[4], 1, 1, 1, 1, dg)
        assert rel_err(y, g(f'{case}.y')) <= TOL
        y.backward(g(f'{case}.go').to(DEV))
        for t, key in zip(ts, ('gx', 'goffset', 'gmask', 'gweight', 'gbias')):
            assert rel_err(t.grad, g(f'{case}.{key}')) <= TOL, key
    finally:
        D.set_default_mode('auto')


@pytest.mark.parametrize('cfg', [
    dict(b=2, c=64, h=20, w=24, co=64, dg=8),                       # relu1_1-like
    dict(b=1, c=128, h=16, w=16, co=128, dg=8),                     # relu2_1-like
    dict(b=1, c=256, h=10, w=12, co=256, dg=8),                     # relu3_1-like
    dict(b=2, c=16, h=9, w=7, co=24, dg=2, off_scale=6.0),          # ragged sizes, many samples out of range
    dict(b=1, c=8, h=6, w=6, co=8, dg=1, groups=2),                 # grouped conv
    dict(b=1, c=8, h=11, w=13, co=4, dg=2, stride=2, pad=2, dil=2),  # stride / dilation
])
@pytest.mark.parametrize('mode', ['fp32', 'auto'])
def test_forward_vs_oracle(cfg, mode):
    cfg = dict(cfg)
    b, c, h, w, co, dg = (cfg.pop(k) for k in ('b', 'c', 'h', 'w', 'co', 'dg'))
    groups, stride, pad, dil = cfg.get('groups', 1), cfg.get('stride', 1), cfg.get('pad', 1), cfg.get('dil', 1)
    x, off, mask, wgt, bias = _rand_problem(b, c, h, w, co, dg, 5, **cfg)
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, stride, pad, dil, groups, dg, dtype=torch.float64)
    out = D.dcn_forward_raw(x.to(DEV), off.to(DEV), mask.to(DEV), wgt.to(DEV), bias.to(DEV), (stride,) * 2, (pad,) * 2,
                            (dil,) * 2, groups, dg, mode=mode)
    assert rel_err(out, ref) <= TOL
    out_nb = D.dcn_forward_raw(x.to(DEV), off.to(DEV), mask.to(DEV), wgt.to(DEV), None, (stride,) * 2, (pad,) * 2,
                               (dil,) * 2, groups, dg, mode=mode)
    assert rel_err(out_nb, ref - bias.double().view(1, -1, 1, 1)) <= TOL


@pytest.mark.parametrize('cfg', [
    dict(b=2, c=32, h=10, w=12, co=32, dg=8),
    dict(b=3, c=16, h=9, w=7, co=24, dg=2, off_scale=6.0),
    dict(b=1, c=8, h=6, w=6, co=8, dg=1, groups=2),
    dict(b=1, c=8, h=11, w=13, co=4, dg=2, stride=2, pad=2, dil=2),
])
def test_backward_vs_oracle(cfg):
    cfg = dict(cfg)
    b, c, h, w, co, dg = (cfg.pop(k) for k in ('b', 'c', 'h', 'w', 'co', 'dg'))
    groups, stride, pad, dil = cfg.get('groups', 1), cfg.get('stride', 1), cfg.get('pad', 1), cfg.get('dil', 1)
    x, off, mask, wgt, bias = _rand_problem(b, c, h, w, co, dg, 9, **cfg)
    ts = [t.to(DEV).requires_grad_(True) for t in (x, off, mask, wgt, bias)]
    y = M.modulated_deform_conv(ts[0], ts[1], ts[2], ts[3], ts[4], stride, pad, dil, groups, dg)
    go = torch.randn(y.shape, generator=torch.Generator().manual_seed(1))
    y.backward(go.to(DEV))
    ref = oracle.modulated_deform_conv_backward_oracle(x, off, mask, wgt, bias, go, stride, pad, dil, groups, dg,
                                                       dtype=torch.float64)
    for t, r, name in zip(ts, ref, ('input', 'offset', 'mask', 'weight', 'bias')):
        assert rel_err(t.grad, r) <= TOL, name


@pytest.mark.parametrize('cfg', [dict(b=3, c=64, h=16, w=24, s=4), dict(b=2, c=128, h=12, w=12, s=2),
                                 dict(b=2, c=256, h=10, w=14, s=1), dict(b=1, c=32, h=8, w=8, s=1, dg=2)])
def test_fused_dynagg_vs_oracle(cfg):
    """Fused DynAgg (conv_out + max_idx -> DCN) against the oracle composition pre_offsets -> glue -> DCN."""
    b, c, h, w, s = (cfg[k] for k in ('b', 'c', 'h', 'w', 's'))
    dg = cfg.get('dg', 8)
    g = torch.Generator().manual_seed(17)
    hc, wc = h // s, w // s
    max_idx = torch.randint(0, (hc - 2) * (wc - 2), (b, hc - 2, wc - 2), generator=g)
    x = torch.randn(b, c, h, w, generator=g)
    conv_out = torch.randn(b, 3 * dg * 9, h, w, generator=g) * 0.7
    wgt = torch.randn(c, c, 3, 3, generator=g) * (c * 9) ** -0.5
    bias = torch.randn(c, generator=g) * 0.1
    key = {1: 'relu3_1', 2: 'relu2_1', 4: 'relu1_1'}[s]
    pre = torch.stack([oracle.pre_offsets_oracle(max_idx[i])[key] for i in range(b)], 0)
    off, mask = oracle.dynagg_offsets_oracle(conv_out, pre, dg)
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, dg, dtype=torch.float64)
    out = D.dynagg_dcn_forward(x.to(DEV), conv_out.to(DEV), max_idx.to(DEV), s, wgt.to(DEV), bias.to(DEV), dg)
    assert rel_err(out, ref) <= TOL
    # and the module-level fast path agrees with the reference-API path
    m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
    m.conv_offset_mask.weight.data.normal_(0, 0.02)
    m.conv_offset_mask.bias.data.normal_(0, 0.3)
    feat = torch.randn(b, c, h, w, generator=g).to(DEV)
    with torch.no_grad():
        y1 = m([x.to(DEV), feat], pre.to(DEV))
        y2 = m.forward_fused([x.to(DEV), feat], max_idx.to(DEV), s)
    assert rel_err(y2, y1) <= TOL


@pytest.mark.parametrize('cfg', [dict(b=2, c=64, h=20, w=24, co=64, dg=8), dict(b=1, c=256, h=10, w=12, co=256, dg=8),
                                 dict(b=3, c=32, h=7, w=5, co=96, dg=2, off_scale=5.0),
                                 dict(b=1, c=64, h=9, w=9, co=32, dg=4, stride=2, pad=1, dil=1)])
def test_tf32_mode_explicit(cfg):
    cfg = dict(cfg)
    b, c, h, w, co, dg = (cfg.pop(k) for k in ('b', 'c', 'h', 'w', 'co', 'dg'))
    stride, pad, dil = cfg.get('stride', 1), cfg.get('pad', 1), cfg.get('dil', 1)
    x, off, mask, wgt, bias = _rand_problem(b, c, h, w, co, dg, 5, **cfg)
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, stride, pad, dil, 1, dg, dtype=torch.float64)
    out = D.dcn_forward_raw(x.to(DEV), off.to(DEV), mask.to(DEV), wgt.to(DEV), bias.to(DEV), (stride,) * 2, (pad,) * 2,
                            (dil,) * 2, 1, dg, mode='tf32')
    assert rel_err(out, ref) <= TOL


def test_tf32_mode_rejects_ineligible():
    x, off, mask, wgt, bias = _rand_problem(1, 8, 6, 6, 8, 2, 1)
    with pytest.raises(RuntimeError):
        D.dcn_forward_raw(x.to(DEV), off.to(DEV), mask.to(DEV), wgt.to(DEV), bias.to(DEV), (1, 1), (1, 1), (1, 1), 1, 2,
                          mode='tf32')


def test_zero_offset_is_plain_conv():
    """Known answer: zero offsets and mask 1 reduce DCNv2 to F.conv2d."""
    x, off, mask, wgt, bias = _rand_problem(2, 32, 12, 12, 16, 4, 3)
    out = D.dcn_forward_raw(x.to(DEV), torch.zeros_like(off).to(DEV), torch.ones_like(mask).to(DEV), wgt.to(DEV),
                            bias.to(DEV), (1, 1), (1, 1), (1, 1), 1, 4)
    ref = torch.nn.functional.conv2d(x.double(), wgt.double(), bias.double(), 1, 1)
    assert rel_err(out, ref) <= TOL


def test_full_size_linearity():
    """BASELINE config 2 large scale (C=64, 160x160): DCN is linear in the input for fixed offsets/mask."""
    b, c, h, w, dg = 2, 64, 160, 160, 8
    x, off, mask, wgt, bias = _rand_problem(b, c, h, w, c, dg, 21, off_scale=8.0)
    x2 = torch.randn(x.shape, generator=torch.Generator().manual_seed(22))
    args = (off.to(DEV), mask.to(DEV), wgt.to(DEV), None, (1, 1), (1, 1), (1, 1), 1, dg)
    ya = D.dcn_forward_raw(x.to(DEV), *args)
    yb = D.dcn_forward_raw(x2.to(DEV), *args)
    yc = D.dcn_forward_raw((2 * x - 3 * x2).to(DEV), *args)
    assert rel_err(yc, 2 * ya - 3 * yb) <= TOL


def test_dynagg_module_golden(golden):
    g = golden('dynagg')
    for case in ('small', 'big_offsets'):
        dg = int(g(f'{case}.dg'))
        c = g(f'{case}.x').shape[1]
        m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
        m.load_state_dict({'weight': g(f'{case}.weight'), 'bias': g(f'{case}.bias'),
                           'conv_offset_mask.weight': g(f'{case}.com_w'), 'conv_offset_mask.bias': g(f'{case}.com_b')})
        x = g(f'{case}.x').to(DEV).requires_grad_(True)
        feat = g(f'{case}.feat').to(DEV).requires_grad_(True)
        y = m([x, feat], g(f'{case}.pre').to(DEV))
        assert rel_err(y, g(f'{case}.y')) <= TOL
        assert m.last_offset_abs_mean() is not None


@pytest.mark.parametrize('fused', [True, False])
def test_dynagg_module_gradients_golden(golden, fused):
    """Backward of DynAgg.forward -- as one autograd node (default) and as the two operator Functions -- against the
    gradients the REFERENCE module produced at the DCN boundary (tests/golden/make_golden.py::gen_dynagg: grad of input,
    weight, bias, offset, mask for the same grad_output), pushed through the glue and the offset convolution in fp64 on
    the host: grad_conv_out = [grad_offset, grad_mask * m * (1 - m)] (ref_mrapa_restoration_arch.py:55-68)."""
    import torch.nn.functional as F
    g = golden('dynagg')
    for case in ('small', 'big_offsets'):
        dg = int(g(f'{case}.dg'))
        c = g(f'{case}.x').shape[1]
        m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
        m.load_state_dict({'weight': g(f'{case}.weight'), 'bias': g(f'{case}.bias'),
                           'conv_offset_mask.weight': g(f'{case}.com_w'), 'conv_offset_mask.bias': g(f'{case}.com_b')})
        m.fused_autograd = fused
        x = g(f'{case}.x').to(DEV).requires_grad_(True)
        feat = g(f'{case}.feat').to(DEV).requires_grad_(True)
        # the offset convolution in exact fp32 like the CPU reference: with cuDNN's TF32 its 1e-3 noise moves a few sampling
        # points across a pixel boundary, where the offset gradient is discontinuous
        old_tf32 = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            y = m([x, feat], g(f'{case}.pre').to(DEV))
            y.backward(g(f'{case}.go').to(DEV))
        finally:
            torch.backends.cudnn.allow_tf32 = old_tf32
        assert rel_err(x.grad, g(f'{case}.gx')) <= TOL
        assert rel_err(m.weight.grad, g(f'{case}.gweight')) <= TOL
        assert rel_err(m.bias.grad, g(f'{case}.gbias')) <= TOL
        mk = g(f'{case}.mask').double()
        g_conv = torch.cat((g(f'{case}.goffset').double(), g(f'{case}.gmask').double() * mk * (1 - mk)), 1)
        f64 = g(f'{case}.feat').double().requires_grad_(True)
        w64 = g(f'{case}.com_w').double().requires_grad_(True)
        b64 = g(f'{case}.com_b').double().requires_grad_(True)
        F.conv2d(f64, w64, b64, 1, 1).backward(g_conv)
        assert rel_err(feat.grad, f64.grad) <= TOL
        assert rel_err(m.conv_offset_mask.weight.grad, w64.grad) <= TOL
        assert rel_err(m.conv_offset_mask.bias.grad, b64.grad) <= TOL


def _dynagg_module_run(fused, bf16, x, feat0, pre, gout, c, dg):
    torch.manual_seed(5)
    m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
    m.conv_offset_mask.weight.data.normal_(0, 0.02)
    m.conv_offset_mask.bias.data.normal_(0, 0.3)
    m.fused_autograd = fused
    feat = feat0.clone().requires_grad_(True)
    f_in = feat
    if bf16:
        m.conv_offset_mask.to(memory_format=torch.channels_last)
        f_in = feat.contiguous(memory_format=torch.channels_last)
    with torch.autocast('cuda', dtype=torch.bfloat16, enabled=bf16):
        y = m([x, f_in], pre)
    y.float().backward(gout)
    assert m.last_offset_abs_mean() is not None
    return (y.float().detach(), feat.grad, m.conv_offset_mask.weight.grad, m.conv_offset_mask.bias.grad, m.weight.grad,
            m.bias.grad)


def test_dynagg_fused_autograd_node_matches_the_two_functions():
    """DynAgg.forward as one autograd node (DynAggDCNFunction) against the reference operator boundaries
    (DynAggOffsetsFunction -> ModulatedDeformConvFunction): same output and the same gradients for the offset
    convolution, the DCN weight / bias and the feature that feeds the offset convolution, in fp32.  Then with the offset
    convolution under bf16 autocast in channels-last (the config-5 training step): there the two-Function path rounds
    offsets / masks and their gradients to bf16 at its boundaries and the fused node does not, and the offset gradient is
    discontinuous across pixel cells, so the check is statistical -- the fused node must be at least as close (relative
    L2) to the fp32 result as the two-Function path is."""
    g = torch.Generator().manual_seed(31)
    b, c, h, w, dg = 2, 64, 20, 24, 8
    x = torch.randn(b, c, h, w, generator=g).to(DEV)
    feat0 = torch.randn(b, c, h, w, generator=g).to(DEV)
    pre = (torch.randn(b, 9, h, w, 2, generator=g) * 2).to(DEV)
    gout = torch.randn(b, c, h, w, generator=g).to(DEV)
    names = ('y', 'g_feat', 'g_com_w', 'g_com_b', 'g_weight', 'g_bias')
    truth = _dynagg_module_run(False, False, x, feat0, pre, gout, c, dg)
    fused32 = _dynagg_module_run(True, False, x, feat0, pre, gout, c, dg)
    for a, r_, name in zip(fused32, truth, names):
        assert a.shape == r_.shape and a.dtype == r_.dtype, name
        assert rel_err(a, r_) <= 1e-5, (name, rel_err(a, r_))

    def rel_l2(a, r_):
        return float((a.double() - r_.double()).norm() / r_.double().norm().clamp_min(1e-30))
    two16 = _dynagg_module_run(False, True, x, feat0, pre, gout, c, dg)
    fused16 = _dynagg_module_run(True, True, x, feat0, pre, gout, c, dg)
    for a, o, r_, name in zip(fused16, two16, truth, names):
        assert a.shape == r_.shape and a.dtype == r_.dtype, name
        e_fused, e_two = rel_l2(a, r_), rel_l2(o, r_)
        assert e_fused <= max(1.25 * e_two, 1e-3) and e_fused <= 0.15, (name, e_fused, e_two)   # bf16 offset conv: ~0.03 px


@pytest.mark.parametrize('bf16', [False, True])
def test_dynagg_node_with_folded_activation(bf16):
    """DynAgg.forward(..., out_slope=0.1, out_like_conv=True): the leaky ReLU that follows DynAgg in MRefSR and the
    hand-off in the offset convolution's dtype / layout as part of the autograd node, against lrelu(DynAgg.forward(...))
    converted afterwards -- same values (the bf16 result is rounded once either way) and the same gradients."""
    g = torch.Generator().manual_seed(41)
    b, c, h, w, dg = 2, 64, 12, 20, 8
    x = torch.randn(b, c, h, w, generator=g).to(DEV)
    feat0 = torch.randn(b, c, h, w, generator=g).to(DEV)
    pre = (torch.randn(b, 9, h, w, 2, generator=g) * 2).to(DEV)
    cl = torch.channels_last
    gout = torch.randn(b, c, h, w, generator=g).to(DEV).contiguous(memory_format=cl)
    res = {}
    for folded in (False, True):
        torch.manual_seed(5)
        m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
        m.conv_offset_mask.weight.data.normal_(0, 0.02)
        m.conv_offset_mask.bias.data.normal_(0, 0.3)
        m.conv_offset_mask.to(memory_format=cl)
        feat = feat0.clone().requires_grad_(True)
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=bf16):
            f_in = feat.contiguous(memory_format=cl)
            if folded:
                y = m([x, f_in], pre, out_slope=0.1, out_like_conv=True)
            else:
                y = torch.nn.functional.leaky_relu(m([x, f_in], pre), 0.1)
                y = y.to(dtype=torch.bfloat16 if bf16 else torch.float32, memory_format=cl)
        assert y.dtype == (torch.bfloat16 if bf16 else torch.float32) and y.is_contiguous(memory_format=cl)
        y.backward(gout.to(y.dtype))
        res[folded] = (y.float().detach(), feat.grad, m.conv_offset_mask.weight.grad, m.weight.grad, m.bias.grad)
    for a, r_, name in zip(res[True], res[False], ('y', 'g_feat', 'g_com_w', 'g_weight', 'g_bias')):
        assert rel_err(a, r_) <= (1e-5 if not bf16 else 1e-5), (name, rel_err(a, r_))


def test_dynagg_glue_golden(golden):
    from mrefsr_b200.dynagg import DynAggOffsetsFunction
    g = golden('dynagg')
    for case in ('small', 'big_offsets'):
        dg = int(g(f'{case}.dg'))
        off, mask = DynAggOffsetsFunction.apply(g(f'{case}.conv_out').to(DEV), g(f'{case}.pre').to(DEV), dg, None)
        assert torch.equal(off.cpu(), g(f'{case}.offset'))
        assert (mask.cpu() - g(f'{case}.mask')).abs().max() <= 1e-6


def test_dcnv1_golden(golden):
    """DCNv1 mirror (DeformConvFunction / deform_conv) against vectors from torchvision's implementation of the
    reference rule, and the three DCNv1 exports of the replaced extension."""
    g = golden('dcnv1')
    dg, groups = int(g('dg')), int(g('groups'))
    ts = [g(k).to(DEV).requires_grad_(True) for k in ('x', 'offset', 'weight')]
    y = M.deform_conv(ts[0], ts[1], ts[2], 1, 1, 1, groups, dg)
    assert rel_err(y, g('y')) <= TOL
    y.backward(g('go').to(DEV))
    for t, key in zip(ts, ('gx', 'goffset', 'gweight')):
        assert rel_err(t.grad, g(key)) <= TOL, key
    x, off, w = (g(k).to(DEV) for k in ('x', 'offset', 'weight'))
    out = torch.empty_like(y)
    e = x.new_empty(0)
    assert D.ext.deform_conv_forward(x, w, off, out, e, e, 3, 3, 1, 1, 1, 1, 1, 1, groups, dg, 2) == 1
    assert rel_err(out, g('y')) <= TOL
    gi, go_ = torch.zeros_like(x), torch.zeros_like(off)
    D.ext.deform_conv_backward_input(x, off, g('go').to(DEV), gi, go_, w, e, 3, 3, 1, 1, 1, 1, 1, 1, groups, dg, 2)
    assert rel_err(gi, g('gx')) <= TOL and rel_err(go_, g('goffset')) <= TOL
    gw = torch.zeros_like(w)
    D.ext.deform_conv_backward_parameters(x, off, g('go').to(DEV), gw, e, e, 3, 3, 1, 1, 1, 1, 1, 1, groups, dg, 1.0, 2)
    assert rel_err(gw, g('gweight')) <= TOL
    m = M.DeformConvPack(8, 12, 3, padding=1, groups=groups, deformable_groups=dg).to(DEV)
    assert sorted(m.state_dict().keys()) == ['conv_offset.bias', 'conv_offset.weight', 'weight']
    assert m(x).shape == (2, 12, 9, 10)


def test_errors():
    x, off, mask, wgt, bias = _rand_problem(1, 8, 6, 6, 8, 2, 1)
    with pytest.raises(NotImplementedError):
        M.modulated_deform_conv(x, off, mask, wgt, bias, 1, 1, 1, 1, 2)           # CPU tensors
    with pytest.raises(RuntimeError):
        M.modulated_deform_conv(x.to(DEV), off.to(DEV), mask.to(DEV), wgt[:, :4].contiguous().to(DEV), bias.to(DEV),
                                1, 1, 1, 1, 2)                                     # channel mismatch


_REF_SO = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref',
                       'deform_conv_ext_ref.so')


def _reference_ext():
    """The reference's own deform_conv_ext, compiled unmodified for sm_100a into oracle/_ref/ by `oracle/build.py --ref`
    where the reference's sources are at hand (checker only), or None."""
    if not os.path.exists(_REF_SO):
        return None
    import importlib.util
    spec = importlib.util.spec_from_file_location('deform_conv_ext_ref', _REF_SO)
    ext = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ext)
    return ext


def _oracle_dcn(x, off, mask, wgt, bias, go, dg=8):
    """fp64 oracle of a 3x3 / stride 1 / pad 1 DCN on CPU tensors: DCNv2 output, its five gradients for grad_output
    `go`, and the DCNv1 output (mask 1, no bias)."""
    f64 = torch.float64
    want = {'output': oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, dg, dtype=f64)}
    grads = oracle.modulated_deform_conv_backward_oracle(x, off, mask, wgt, bias, go, 1, 1, 1, 1, dg, dtype=f64)
    want.update(zip(('input', 'offset', 'mask', 'weight', 'bias'), grads))
    want['dcnv1'] = oracle.modulated_deform_conv_oracle(x, off, torch.ones_like(mask), wgt, None, 1, 1, 1, 1, dg, dtype=f64)
    return want


def _drive_ext(ext, x, off, mask, wgt, bias, go, grad_weight_init=0.0, grad_bias_init=0.0):
    """Call a deform_conv_ext module the way basicsr/ops/dcn/deform_conv.py:147-170 does (caller-allocated output, size-0
    `ones` / `columns` scratch, zero-initialised input / offset / mask gradients; grad_weight / grad_bias start at the
    given values).  Returns the results keyed like _oracle_dcn, and deform_conv_forward's return value."""
    empty = x.new_empty(0)
    got = {'output': x.new_empty(x.shape[0], wgt.shape[0], *x.shape[2:])}   # 3x3, stride 1, pad 1
    ext.modulated_deform_conv_forward(x, wgt, bias, empty, off, mask, got['output'], empty, 3, 3, 1, 1, 1, 1, 1, 1, 1, 8,
                                      True)
    g = [torch.zeros_like(t) for t in (x, wgt, bias, off, mask)]
    g[1].fill_(grad_weight_init)
    g[2].fill_(grad_bias_init)
    ext.modulated_deform_conv_backward(x, wgt, bias, empty, off, mask, empty, g[0], g[1], g[2], g[3], g[4], go, 3, 3, 1,
                                       1, 1, 1, 1, 1, 1, 8, True)
    got.update(zip(('input', 'weight', 'bias', 'offset', 'mask'), g))
    got['dcnv1'] = torch.empty_like(got['output'])
    rc = ext.deform_conv_forward(x, wgt, off, got['dcnv1'], empty, empty, 3, 3, 1, 1, 1, 1, 1, 1, 1, 8, 2)
    return got, rc


def test_against_reference_cuda_extension():
    """The product DCN (dcn_forward_raw, dcn_backward_raw, deform_conv) on a problem with many samples at and beyond the
    image border (offsets ~ N(0, 4^2)): against the fp64 oracle, and, where oracle/_ref holds the reference's own
    deform_conv_ext, against the reference's kernels on the same inputs."""
    cpu = _rand_problem(2, 64, 24, 20, 64, 8, 31, off_scale=4.0)
    go = torch.randn(2, 64, 24, 20, generator=torch.Generator().manual_seed(3))
    want = _oracle_dcn(*cpu, go)
    x, off, mask, wgt, bias, go = (t.to(DEV) for t in cpu + (go,))
    got = {'output': D.dcn_forward_raw(x, off, mask, wgt, bias, (1, 1), (1, 1), (1, 1), 1, 8)}
    got.update(zip(('input', 'offset', 'mask', 'weight', 'bias'),
                   D.dcn_backward_raw(x, off, mask, wgt, go, (1, 1), (1, 1), (1, 1), 1, 8, True)))
    got['dcnv1'] = M.deform_conv(x, off, wgt, 1, 1, 1, 1, 8)
    for name in want:
        assert rel_err(got[name], want[name]) <= TOL, name
    ref = _reference_ext()
    if ref is not None:
        ref_got, _ = _drive_ext(ref, x, off, mask, wgt, bias, go)
        for name in ref_got:
            assert rel_err(got[name], ref_got[name]) <= TOL, ('reference extension', name)


def test_torch_extension_module_is_call_compatible_with_the_reference_extension():
    """mrefsr_b200/torch_ext/deform_conv_ext.so -- the pybind module that replaces the reference's deform_conv_ext build
    (csrc/torch_ext/deform_conv_ext.cpp) -- driven with the reference's argument lists, grad_weight / grad_bias
    accumulated into (deform_conv_cuda.cpp:571-685): against the fp64 oracle, and, where oracle/_ref holds the
    reference's own deform_conv_ext, against the reference driven with the same calls."""
    from mrefsr_b200 import build as B
    ours = B.load_torch_ext()
    cpu = _rand_problem(2, 64, 24, 20, 64, 8, 33, off_scale=3.0)
    go = torch.randn(2, 64, 24, 20, generator=torch.Generator().manual_seed(2))
    want = _oracle_dcn(*cpu, go)
    want['weight'] = want['weight'] + 0.5                    # pre-existing content: grad_weight / grad_bias accumulate
    want['bias'] = want['bias'] - 1.0
    x, off, mask, wgt, bias, go = (t.to(DEV) for t in cpu + (go,))
    got, rc = _drive_ext(ours, x, off, mask, wgt, bias, go, 0.5, -1.0)
    assert rc == 1                                           # DCNv1 export: the reference's int return value
    for name in want:
        assert rel_err(got[name], want[name]) <= TOL, name
    ref = _reference_ext()
    if ref is not None:
        ref_got, _ = _drive_ext(ref, x, off, mask, wgt, bias, go, 0.5, -1.0)
        for name in ref_got:
            assert rel_err(got[name], ref_got[name]) <= TOL, ('reference extension', name)
    # fp16 tensors are accepted like the reference's AT_DISPATCH_FLOATING_TYPES_AND_HALF (computed in fp32 here)
    empty = x.new_empty(0)
    oh = x.new_empty(2, 64, 24, 20).half()
    ours.modulated_deform_conv_forward(x.half(), wgt.half(), bias.half(), empty, off.half(), mask.half(), oh, empty, 3, 3,
                                       1, 1, 1, 1, 1, 1, 1, 8, True)
    assert rel_err(oh.float(), want['output']) <= 2e-2
    # the reference's error behaviour: kernel-shape mismatch -> RuntimeError
    with pytest.raises(RuntimeError, match="kernel shape won't match"):
        ours.modulated_deform_conv_forward(x, wgt, bias, empty, off, mask, x.new_empty(2, 64, 24, 20), empty, 5, 5, 1, 1, 1,
                                           1, 1, 1, 1, 8, True)


def test_dynagg_dcn_forward_into_several_buffers():
    """Epilogue of the reference-sharded mode: every tile stored to each destination buffer, at the global reference
    slot of the gathered [n, R, C, H, W] tensor (here two local buffers stand in for the peers' copies)."""
    from mrefsr_b200.dcn import dynagg_dcn_forward, dynagg_dcn_forward_into
    g = torch.Generator().manual_seed(21)
    n, r_local, R, lo, c, hw, dg, s = 2, 3, 8, 4, 64, 16, 8, 1
    b = n * r_local
    x = torch.randn(b, c, hw, hw, generator=g).to(DEV)
    conv_out = torch.randn(b, 3 * dg * 9, hw, hw, generator=g).to(DEV)
    hp = hw // s - 2
    max_idx = torch.randint(0, hp * hp, (b, hp, hp), generator=g).to(DEV)
    wgt = (torch.randn(c, c, 3, 3, generator=g) * 0.05).to(DEV)
    bias = torch.randn(c, generator=g).to(DEV)
    want = dynagg_dcn_forward(x, conv_out, max_idx, s, wgt, bias, dg).view(n, r_local, c, hw, hw)
    bufs = [torch.full((n, R, c, hw, hw), -7.0, device=DEV) for _ in range(2)]
    dynagg_dcn_forward_into(x, conv_out, max_idx, s, wgt, bias, dg, [t.data_ptr() for t in bufs], r_local, R, lo)
    torch.cuda.synchronize()
    for t in bufs:
        assert torch.equal(t[:, lo:lo + r_local], want)
        assert bool((t[:, :lo] == -7.0).all()) and bool((t[:, lo + r_local:] == -7.0).all())   # other slots untouched


def test_dynagg_dcn_forward_into_pixel_slabs():
    """Pixel-slab routing of the reference-sharded mode: output row oy is stored to buffer oy // slab_rows only, at
    the global reference slot; four local buffers stand in for four ranks.  Reassembling the slabs must give exactly
    the plain forward, and nothing else may be written."""
    from mrefsr_b200.dcn import dynagg_dcn_forward, dynagg_dcn_forward_into
    g = torch.Generator().manual_seed(22)
    n, r_local, R, lo, c, h, w, dg, s, ranks = 1, 2, 8, 4, 64, 32, 48, 8, 2, 4
    b = n * r_local
    x = torch.randn(b, c, h, w, generator=g).to(DEV)
    conv_out = torch.randn(b, 3 * dg * 9, h, w, generator=g).to(DEV)
    hp, wp = h // s - 2, w // s - 2
    max_idx = torch.randint(0, hp * wp, (b, hp, wp), generator=g).to(DEV)
    wgt = (torch.randn(c, c, 3, 3, generator=g) * 0.05).to(DEV)
    bias = torch.randn(c, generator=g).to(DEV)
    want = dynagg_dcn_forward(x, conv_out, max_idx, s, wgt, bias, dg).view(r_local, n, c, h, w).transpose(0, 1)
    hs = h // ranks
    bufs = [torch.full((n, R, c, hs, w), -7.0, device=DEV) for _ in range(ranks)]
    dynagg_dcn_forward_into(x, conv_out, max_idx, s, wgt, bias, dg, [t.data_ptr() for t in bufs], r_local, R, lo,
                            slab_rows=hs)
    torch.cuda.synchronize()
    for k, t in enumerate(bufs):
        assert torch.equal(t[:, lo:lo + r_local], want[:, :, :, k * hs:(k + 1) * hs])
        assert bool((t[:, :lo] == -7.0).all()) and bool((t[:, lo + r_local:] == -7.0).all())


@pytest.mark.parametrize('scale', [1.0, 3e5, 1e-6, float('inf')])
@pytest.mark.parametrize('nhwc', [False, True])
def test_input_dynamic_range(scale, nhwc):
    """The tcgen05 path keeps fp32's exponent range end to end (fp32 staging copy, TF32 operands): inputs scaled far
    outside fp16's range must come out as accurate as O(1) inputs, and Inf must propagate to exactly the outputs the
    reference formula makes non-finite.  (Guards the rejected fp16-staging experiment of profiles/r01s_dcn_ab.md
    against coming back without a range check.)"""
    b, c, h, w, co, dg = 2, 64, 12, 16, 64, 8
    x, off, mask, wgt, bias = _rand_problem(b, c, h, w, co, dg, 11)
    bias = torch.zeros_like(bias)
    if scale == float('inf'):
        x = x.clone()
        x[0, 3, 5, 7] = float('inf')
        xs = x
    else:
        xs = x * scale
    ref = oracle.modulated_deform_conv_oracle(xs, off, mask, wgt, bias, 1, 1, 1, 1, dg, dtype=torch.float64)
    xd = xs.to(DEV)
    if nhwc:
        # the channels-last entry point: raw conv_offset_mask output + arg-max map; zero flow, so that
        # offset = conv_out[:, :144], mask = sigmoid(conv_out[:, 144:])
        conv_out = torch.cat([off, torch.logit(mask.clamp(1e-4, 1 - 1e-4))], 1)
        ref = oracle.modulated_deform_conv_oracle(xs, off, mask.clamp(1e-4, 1 - 1e-4), wgt, bias, 1, 1, 1, 1, dg,
                                                  dtype=torch.float64)
        ys, xg = torch.meshgrid(torch.arange(h - 2), torch.arange(w - 2), indexing='ij')
        idx = (ys * (w - 2) + xg).expand(b, -1, -1).contiguous().to(DEV)
        out = D.dynagg_dcn_forward(xd.contiguous(memory_format=torch.channels_last), conv_out.to(DEV), idx, 1,
                                   wgt.to(DEV), bias.to(DEV), dg)
    else:
        out = D.dcn_forward_raw(xd, off.to(DEV), mask.to(DEV), wgt.to(DEV), bias.to(DEV), (1, 1), (1, 1), (1, 1), 1, dg,
                                mode='tf32')
    if scale == float('inf'):
        bad_ref, bad = ~torch.isfinite(ref), ~torch.isfinite(out.cpu())
        assert bad_ref.any() and torch.equal(bad, bad_ref)
        ok = ~bad_ref
        assert float((out.cpu().double() - ref)[ok].abs().max() / ref[ok].abs().max()) <= TOL
    else:
        assert rel_err(out, ref) <= TOL


@pytest.mark.parametrize('cfg', [dict(b=3, c=64, h=48, w=64, s=4), dict(b=2, c=128, h=40, w=48, s=2),
                                 dict(b=2, c=256, h=24, w=40, s=1), dict(b=2, c=64, h=75, w=75, s=1)])
@pytest.mark.parametrize('flow', ['translate', 'piecewise', 'border'])
def test_coherent_and_border_flows_vs_oracle(cfg, flow):
    """Fused DynAgg + DCNv2 and the operator entry point against the oracle on the flows of real reference images,
    with a few large learned offsets on top: a common translation + small learned residual ('translate'), two regions
    with different translations ('piecewise': tiles on the seam sample from both), and translations that push most
    sampling points over the image border ('border': corners outside the plane contribute 0,
    deform_conv_cuda_kernel.cu:468-497).  1 / 2 / 4 deform groups per 32-channel slab; the 75 x 75 grid takes the
    linear row mapping of the CTA tiles, the others square patches."""
    b, c, h, w, s = (cfg[k] for k in ('b', 'c', 'h', 'w', 's'))
    dg = 8
    g = torch.Generator().manual_seed(31)
    hc, wc = h // s, w // s
    hp, wp = hc - 2, wc - 2
    ys, xs = torch.meshgrid(torch.arange(hp), torch.arange(wp), indexing='ij')
    idx = []
    for i in range(b):
        if flow == 'translate':
            dy, dx = (2, -1) if i % 2 == 0 else (-1, 3)
            m = (ys + dy).clamp(0, hp - 1) * wp + (xs + dx).clamp(0, wp - 1)
        elif flow == 'piecewise':
            left = (ys + 1).clamp(0, hp - 1) * wp + (xs + 2).clamp(0, wp - 1)
            right = (ys - 2).clamp(0, hp - 1) * wp + (xs - 1).clamp(0, wp - 1)
            m = torch.where(xs < wp // 2 + i, left, right)
        else:
            dy, dx = (hp - 2, wp - 2) if i % 2 == 0 else (-(hp - 2), -(wp - 2))
            m = (ys + dy).clamp(0, hp - 1) * wp + (xs + dx).clamp(0, wp - 1)
        idx.append(m)
    max_idx = torch.stack(idx)
    x = torch.randn(b, c, h, w, generator=g)
    conv_out = torch.randn(b, 3 * dg * 9, h, w, generator=g) * 0.6
    conv_out[:, :2 * dg * 9, ::7, ::5] *= 8          # a few large learned offsets
    wgt = torch.randn(c, c, 3, 3, generator=g) * (c * 9) ** -0.5
    bias = torch.randn(c, generator=g) * 0.1
    key = {1: 'relu3_1', 2: 'relu2_1', 4: 'relu1_1'}[s]
    pre = torch.stack([oracle.pre_offsets_oracle(max_idx[i])[key] for i in range(b)], 0)
    off, mask = oracle.dynagg_offsets_oracle(conv_out, pre, dg)
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, dg, dtype=torch.float64)
    out = D.dynagg_dcn_forward(x.to(DEV), conv_out.to(DEV), max_idx.to(DEV), s, wgt.to(DEV), bias.to(DEV), dg)
    assert rel_err(out, ref) <= TOL
    # the operator entry point with the same (materialised) offsets
    out2 = D.dcn_forward_raw(x.to(DEV), off.to(DEV), mask.to(DEV), wgt.to(DEV), bias.to(DEV), (1, 1), (1, 1), (1, 1), 1,
                             dg, mode='tf32')
    assert rel_err(out2, ref) <= TOL


@pytest.mark.parametrize('cfg', [dict(b=2, c=64, hw=160, s=4), dict(b=1, c=128, hw=150, s=2), dict(b=1, c=64, hw=300, s=4),
                                 dict(b=1, c=256, hw=75, s=1), dict(b=1, c=128, hw=256, s=2)])
def test_native_grids_vs_oracle(cfg):
    """Fused DynAgg + DCNv2 at the grids of the BASELINE configurations: 160^2 (config 2, large scale), 75 / 150 / 300
    (config 3: LMR 300x300, incl. the 75-wide grid that the 256-row kernel maps linearly because patches would pad it
    by 14 %), 256^2 (config 4's middle scale), against the plain-C oracle (oracle/dcn_ref.c, OpenMP) fed with the
    oracle's own pre-offsets and DynAgg glue."""
    from oracle.dcn import modulated_deform_conv_c
    b, c, hw, s = (cfg[k] for k in ('b', 'c', 'hw', 's'))
    dg = 8
    g = torch.Generator().manual_seed(hw + c)
    hc = hw // s
    hp = hc - 2
    ys, xs = torch.meshgrid(torch.arange(hp), torch.arange(hp), indexing='ij')
    coherent = (ys + 3).clamp(0, hp - 1) * hp + (xs - 2).clamp(0, hp - 1)
    rnd = torch.randint(0, hp * hp, (hp, hp), generator=g)
    max_idx = torch.stack([torch.where(xs < hp // 2, coherent, rnd) for _ in range(b)])   # half translation, half random
    x = torch.randn(b, c, hw, hw, generator=g)
    conv_out = torch.randn(b, 3 * dg * 9, hw, hw, generator=g) * 0.5
    wgt = torch.randn(c, c, 3, 3, generator=g) * (c * 9) ** -0.5
    bias = torch.randn(c, generator=g) * 0.1
    key = {1: 'relu3_1', 2: 'relu2_1', 4: 'relu1_1'}[s]
    pre = torch.stack([oracle.pre_offsets_oracle(max_idx[i])[key] for i in range(b)], 0)
    off, mask = oracle.dynagg_offsets_oracle(conv_out, pre, dg)
    ref = modulated_deform_conv_c(x, off, mask, wgt, bias, 1, 1, 1, 1, dg)
    out = D.dynagg_dcn_forward(x.to(DEV), conv_out.to(DEV), max_idx.to(DEV), s, wgt.to(DEV), bias.to(DEV), dg)
    torch.cuda.synchronize()
    assert rel_err(out, ref) <= TOL


@pytest.mark.parametrize('shape', [dict(M=576, N=1600, K=64, batch=3), dict(M=130, N=70, K=36, batch=2),
                                   dict(M=2304, N=6400, K=256, batch=1), dict(M=64, N=576, K=25600, batch=2, reduce=True, splits=30),
                                   dict(M=256, N=2304, K=1600, batch=5, reduce=True, splits=4),
                                   dict(M=96, N=200, K=100, batch=3, reduce=True, splits=7)])
def test_backward_gemm_on_tcgen05(shape):
    """csrc/gemm_tc.cu, the GEMM behind both products of the DCN backward (deform_conv_cuda.cpp:623-626, :659-664),
    through its C-ABI test entry against torch in fp64: TF32 operands, fp32 accumulation -> 1e-3 of the result's
    scale.  Ragged tiles (M, N, K not multiples of the 128 x 128 x 32 tile), a shared A operand, and the split-K
    reduce mode whose partial sums must add up to the batch-summed product."""
    from mrefsr_b200 import _lib
    M_, N_, K_, batch = (shape[k] for k in ('M', 'N', 'K', 'batch'))
    reduce, splits = shape.get('reduce', False), shape.get('splits', 1)
    g = torch.Generator().manual_seed(M_ + N_)
    lda = (K_ + 3) // 4 * 4 + 4                      # pitches larger than K: padding columns must never be read as data
    a = torch.randn(batch if reduce else 1, M_, lda, generator=g).to(DEV)
    b = torch.randn(batch, N_, lda, generator=g).to(DEV)
    n_out = splits if reduce else batch
    ldd = N_ + 3
    d = torch.full((n_out, M_, ldd), float('nan'), device=DEV)
    rc = _lib.lib().mrefsr_gemm_tf32_nt(_lib.ptr(a), lda, M_ * lda if reduce else 0, _lib.ptr(b), lda, N_ * lda, _lib.ptr(d), ldd,
                                        M_ * ldd, M_, N_, K_, batch, int(reduce), splits, _lib.stream_ptr(a.device))
    _lib.check(rc, 'mrefsr_gemm_tf32_nt')
    torch.cuda.synchronize()
    a64, b64 = a[..., :K_].double().cpu(), b[..., :K_].double().cpu()
    assert torch.isnan(d[..., N_:]).all()             # nothing written beyond the N columns
    if reduce:
        ref = torch.einsum('zmk,znk->mn', a64, b64)
        out = d[..., :N_].double().cpu().sum(0)
    else:
        ref = torch.einsum('mk,znk->zmn', a64[0], b64)
        out = d[..., :N_].double().cpu()
    assert float((out - ref).abs().max() / ref.abs().max()) <= 1e-3


def test_explicitly_packed_weights_give_the_same_bits():
    """`pack_weight` + `weight_packed=` (a caller with frozen weights packs once) against the per-call repack; a packed
    tensor of the wrong shape is refused."""
    g = torch.Generator().manual_seed(3)
    b, c, hw, dg, s = 2, 64, 16, 8, 1
    x = torch.randn(b, c, hw, hw, generator=g).to(DEV)
    conv_out = (torch.randn(b, 216, hw, hw, generator=g) * 0.5).to(DEV)
    idx = torch.randint(0, (hw - 2) ** 2, (b, hw - 2, hw - 2), generator=g).to(DEV)
    bias = torch.zeros(c, device=DEV)
    w = (torch.randn(c, c, 3, 3, generator=g) * 0.05).to(DEV)
    y0 = D.dynagg_dcn_forward(x, conv_out, idx, s, w, bias, dg)
    y1 = D.dynagg_dcn_forward(x, conv_out, idx, s, w, bias, dg, weight_packed=D.pack_weight(w))
    assert torch.equal(y0, y1)
    with pytest.raises(RuntimeError):
        D.dynagg_dcn_forward(x, conv_out, idx, s, w, bias, dg, weight_packed=torch.zeros(c, 8 * c, device=DEV))


@pytest.mark.parametrize('hw', [(12, 16), (7, 9), (40, 40), (5, 4)])
def test_dynagg_glue_both_kernels_vs_oracle(hw):
    """DynAgg offset / mask assembly (ref_mrapa_restoration_arch.py:55-73): the four-positions-per-thread kernel
    (h*w % 4 == 0) and the scalar one (other sizes) against the oracle, offsets bit-exact, and the mean-|learned offset|
    statistic the reference computes with a host sync (:70-71)."""
    from mrefsr_b200.dynagg import DynAggOffsetsFunction
    h, w = hw
    b, dg, k = 3, 8, 9
    g = torch.Generator().manual_seed(h * w)
    conv_out = torch.randn(b, 3 * dg * k, h, w, generator=g)
    pre = torch.randint(-20, 21, (b, k, h, w, 2), generator=g).float()
    stats = torch.zeros(1, device=DEV)
    off, mask = DynAggOffsetsFunction.apply(conv_out.to(DEV), pre.to(DEV), dg, stats)
    o_off, o_mask = oracle.dynagg_offsets_oracle(conv_out, pre, dg)
    assert torch.equal(off.cpu(), o_off)
    assert (mask.cpu() - o_mask).abs().max() <= 1e-6
    want = float(conv_out[:, :2 * dg * k].abs().double().sum())
    assert abs(float(stats.item()) - want) <= 1e-4 * want
