"""The fused DynAgg backward (mrefsr_dynagg_dcn_backward, DynAggFusedFunction, DynAgg.forward_fused under autograd):
gradients read from the raw conv_offset_mask output and the matcher's arg-max map, against the fp64 oracle
(pre_offsets_oracle -> dynagg_offsets_oracle -> modulated_deform_conv_backward_oracle with the reference's fp32
sampling positions) and against the materialised node DynAggDCNFunction fed the pre-offsets of the same map."""
import contextlib

import pytest
import torch

import mrefsr_b200 as M
import oracle
from mrefsr_b200 import _lib
from mrefsr_b200 import dcn as D
from mrefsr_b200 import trunk as T
from mrefsr_b200.dynagg import DynAggDCNFunction, DynAggFusedFunction
from oracle.dcn import sampling_positions
from tests.test_dcn_backward_gpu import _assert_kernels, _border_sets, _oracle, _traced
from tests.util import rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 1e-3
CL = torch.channels_last
_LAYER = {1: 'relu3_1', 2: 'relu2_1', 4: 'relu1_1'}


@contextlib.contextmanager
def _mode(mode):
    D.set_default_mode(mode)
    try:
        yield
    finally:
        D.set_default_mode('auto')


def _ran(names, *subs):
    """some kernel of the trace has all the substrings (the sample source is the type of its last parameter)"""
    return any(all(sub in n for sub in subs) for n in names)


def _problem(b, c, h, w, dg, s, seed, kind='random', device='cpu'):
    """(x, conv_out, max_idx, weight, bias, grad_output).  kind 'random': learned offsets ~ N(0, 1.5^2) and arg-max
    entries anywhere on the grid; 'integer': zero learned offsets and zero mask logits (DynAgg at initialisation) with
    arg-max entries on the grid border, so that points land exactly on rows / columns -1, 0, H-1, H; 'fractional': the
    same flows plus learned offsets in (-1, 1), which puts points into (-1, 0) and (H-1, H)."""
    g = torch.Generator().manual_seed(seed)
    hp, wp = h // s - 2, w // s - 2
    x = torch.randn(b, c, h, w, generator=g)
    co = torch.randn(b, 3 * dg * 9, h, w, generator=g)
    co[:, :2 * dg * 9] *= 1.5
    if kind == 'random':
        mi = torch.randint(0, hp * wp, (b, hp, wp), generator=g)
    else:
        my = torch.tensor([0, hp - 1])[torch.randint(0, 2, (b, hp, wp), generator=g)]
        mx = torch.tensor([0, wp - 1])[torch.randint(0, 2, (b, hp, wp), generator=g)]
        inner = torch.rand(b, hp, wp, generator=g) < 0.3
        my = torch.where(inner, torch.randint(0, hp, (b, hp, wp), generator=g), my)
        mi = my * wp + mx
        if kind == 'integer':
            co.zero_()
        else:       # half the points: a fraction in (-0.95, 0.95) off the integer position
            frac = torch.rand(b, 2 * dg * 9, h, w, generator=g) * 1.9 - 0.95
            co[:, :2 * dg * 9] = torch.where(torch.rand(frac.shape, generator=g) < 0.5, frac, torch.zeros(()))
            co[:, 2 * dg * 9:] = 0
    wgt = torch.randn(c, c, 3, 3, generator=g) * (c * 9) ** -0.5
    bias = torch.randn(c, generator=g) * 0.1
    go = torch.randn(b, c, h, w, generator=g)
    return tuple(t.to(device) for t in (x, co, mi, wgt, bias, go))


def _materialised(co, mi, s, dg):
    """(offset, mask) of the oracle glue fed the oracle pre-offsets of max_idx at flow scale s (fp32, CPU)."""
    pre = torch.stack([oracle.pre_offsets_oracle(mi[i].cpu())[_LAYER[s]] for i in range(mi.shape[0])])
    return oracle.dynagg_offsets_oracle(co.cpu(), pre, dg)


def _want(x, co, mi, wgt, bias, go, s, dg):
    """oracle (grad_input, grad_conv_out, grad_weight, grad_bias) and the border subsets of grad_offset / grad_input."""
    off, mask = _materialised(co, mi, s, dg)
    gi, goff, gm, gw, gb = _oracle(x.cpu(), off, mask, wgt.cpu(), bias.cpu(), go.cpu(), 3, 1, 1, 1, 1, dg)
    m = mask.double()
    return (gi, torch.cat((goff, gm * m * (1 - m)), 1), gw, gb), _border_sets(off, x.shape[2], x.shape[3], x.shape[1], 3, 1,
                                                                               1, 1, dg), off


def _raw(x, co, mi, s, wgt, go, dg, cl=False, **kw):
    xin = x.contiguous(memory_format=CL) if cl else x
    return D.dynagg_dcn_backward_raw(xin, co, mi, s, wgt, go, dg, True, **kw)


def _check(got, want, sets, dg, what):
    for name, g, r in zip(('input', 'conv_out', 'weight', 'bias'), got, want):
        assert g is not None and g.shape == r.shape, (what, name)
        assert rel_err(g, r) <= TOL, (what, name, rel_err(g, r))
    off_sel, in_sel = sets
    b, _, h, w = got[1].shape
    g_off = got[1][:, :2 * dg * 9].detach().cpu()
    assert rel_err(g_off[off_sel], want[1][:, :2 * dg * 9][off_sel]) <= TOL, (what, 'conv_out (border subset)')
    assert rel_err(got[0].detach().cpu()[in_sel], want[0][in_sel]) <= TOL, (what, 'input (border subset)')


_SHAPES = {
    'c64_s4': dict(b=2, c=64, h=32, w=32, dg=8, s=4),
    'c128_s2': dict(b=2, c=128, h=24, w=28, dg=8, s=2),
    'c256_s1': dict(b=2, c=256, h=12, w=14, dg=8, s=1),
    'grid75_no_tma': dict(b=1, c=64, h=75, w=75, dg=8, s=1),        # 5625 positions: the planar im2col + SIMT grad_weight
    'dg2_16ch': dict(b=2, c=32, h=16, w=20, dg=2, s=2),
    'dg2_32ch': dict(b=2, c=64, h=12, w=16, dg=2, s=1),
}


@pytest.mark.parametrize('layout', ['nchw', 'channels_last'])
@pytest.mark.parametrize('case', list(_SHAPES))
def test_fused_backward_vs_oracle(case, layout):
    p = _SHAPES[case]
    b, c, h, w, dg, s = (p[k] for k in ('b', 'c', 'h', 'w', 'dg', 's'))
    x, co, mi, wgt, bias, go = _problem(b, c, h, w, dg, s, 100 + c + s, device=DEV)
    want, sets, _ = _want(x, co, mi, wgt, bias, go, s, dg)
    cl = layout == 'channels_last'
    got, names = _traced(lambda: _raw(x, co, mi, s, wgt, go, dg, cl=cl))
    if cl:
        assert got[0].is_contiguous(memory_format=CL)
    _check(got, want, sets, dg, case + ' ' + layout)
    if case == 'grid75_no_tma':
        assert _ran(names, 'coord_nhwc', 'DynAggSrc') and _ran(names, 'im2col_kernel(', 'DynAggSrc'), case
        _assert_kernels(names, ['bwd_weight'], ['coord_cols', 'im2col_planes'], case)
    else:
        assert _ran(names, 'coord_cols_kernel<false>', 'DynAggSrc'), case
    # the input's NCHW -> NHWC copy runs for NCHW x only (the other one is grad_output's)
    _assert_kernels(names, [('nchw_to_nhwc', 1 if cl else 2)], ('PlaneSrc', 'dynagg_offsets', 'pre_offsets'), case)
    if cl:      # the same gradients as from the NCHW input, grad_input transposed
        ref = _raw(x, co, mi, s, wgt, go, dg)
        assert torch.equal(got[1], ref[1])
        for i in (0, 2, 3):     # grad_input / the SIMT grad_weight / grad_bias are summed with atomics
            assert rel_err(got[i], ref[i]) <= 1e-6, (i, rel_err(got[i], ref[i]))


@pytest.mark.parametrize('kind', ['integer', 'fractional'])
def test_integer_and_border_positions(kind):
    b, c, h, w, dg, s = 2, 64, 24, 20, 8, 1
    x, co, mi, wgt, bias, go = _problem(b, c, h, w, dg, s, 7, kind=kind, device=DEV)
    want, sets, off = _want(x, co, mi, wgt, bias, go, s, dg)
    hy, wx = sampling_positions(off.double(), 3, 3, (1, 1), (1, 1), (1, 1), dg, torch.float64, fp32_positions=True)
    for t, n in ((hy, h), (wx, w)):
        for v in (-1, 0, n - 1, n):
            assert bool((t == v).any()), (kind, v)
    if kind == 'fractional':
        assert bool(((hy > -1) & (hy < 0)).any()) and bool(((hy > h - 1) & (hy < h)).any())
    _check(_raw(x, co, mi, s, wgt, go, dg), want, sets, dg, kind)


def _materialised_node(x, co, mi, s, wgt, bias, dg, go, fused, **kw):
    """(output, grad_conv_out, grad_weight, grad_bias) of one node, materialised (DynAggDCNFunction fed
    pre_offsets(max_idx)) or fused (DynAggFusedFunction)."""
    cot, wt, bt = (t.clone().requires_grad_(True) for t in (co, wgt, bias))
    stats = torch.zeros(1, device=DEV)
    if fused:
        y = DynAggFusedFunction.apply(x, cot, mi, s, wt, bt, dg, *kw.values())
    else:
        pre = M.pre_offsets(mi, scales=(s,))[0]
        y = DynAggDCNFunction.apply(x, cot, pre, wt, bt, dg, stats, *kw.values())
    y.backward(go.to(y.dtype))
    return y.detach(), cot.grad, wt.grad, bt.grad


@pytest.mark.parametrize('mode', ['tf32', 'tf32x3'])
@pytest.mark.parametrize('s', [1, 2, 4])
def test_same_positions_as_the_materialised_node(s, mode):
    """The sampling positions are the same fp32 sums, so no point changes cell: the gradients agree with the
    materialised node up to the mask's sigmoid (__expf here, expf there).  In 'tf32' mode a last-bit difference of a
    mask can move a gathered sample * mask across a tf32 rounding boundary of the GEMM operands, so the output and
    grad_weight are held to 1e-3 there; grad_conv_out and grad_bias do not pass through a tf32 operand."""
    c = {1: 256, 2: 128, 4: 64}[s]
    x, co, mi, wgt, bias, go = _problem(2, c, 8 * s, 10 * s, 8, s, 50 + s, device=DEV)
    with _mode(mode):
        a = _materialised_node(x, co, mi, s, wgt, bias, 8, go, fused=False)
        f = _materialised_node(x, co, mi, s, wgt, bias, 8, go, fused=True)
    for name, u, v in zip(('output', 'conv_out', 'weight', 'bias'), f, a):
        tol = 1e-3 if mode == 'tf32' and name in ('output', 'weight') else 1e-5
        assert rel_err(u, v) <= tol, (s, mode, name, rel_err(u, v))


def test_chunk_rounds_at_the_training_shape():
    """B 20, C 64, 160^2 (flow scale 4): the 1 GiB chunk loop runs rounds of 18 + 2 samples.  A dense call equals the two
    single-round sub-batch calls: grad_conv_out bit for bit, grad_weight up to the order of the split-K sums."""
    b, nb, dg, s = 20, 18, 8, 4
    x, co, mi, wgt, bias, go = _problem(b, 64, 160, 160, dg, s, 77, device=DEV)
    kw = dict(need_input=False)
    n0 = _lib.launch_count()
    full = _raw(x, co, mi, s, wgt, go, dg, **kw)
    torch.cuda.synchronize()
    n_dense = _lib.launch_count() - n0
    parts = []
    for lo, hi in ((0, nb), (nb, b)):
        n0 = _lib.launch_count()
        parts.append(_raw(*(t[lo:hi].contiguous() for t in (x, co, mi)), s, wgt, go[lo:hi].contiguous(), dg, **kw))
        torch.cuda.synchronize()
        # a round: columns GEMM, coordinate + columns kernel, grad_weight GEMM, split-K sum
        assert n_dense - (_lib.launch_count() - n0) == 4, (n_dense, _lib.launch_count() - n0)
    assert torch.equal(full[1][:nb], parts[0][1]) and torch.equal(full[1][nb:], parts[1][1])
    gw_sum = parts[0][2].double() + parts[1][2].double()
    assert rel_err(full[2], gw_sum) <= 1e-4, rel_err(full[2], gw_sum)
    assert rel_err(full[3], parts[0][3].double() + parts[1][3].double()) <= 1e-4


def test_backward_is_deterministic():
    x, co, mi, wgt, bias, go = _problem(3, 64, 40, 48, 8, 4, 21, device=DEV)
    a = _raw(x, co, mi, 4, wgt, go, 8)
    b = _raw(x, co, mi, 4, wgt, go, 8)
    for i in (1, 2):
        assert torch.equal(a[i], b[i]), i
    assert rel_err(a[3], b[3]) <= 1e-6       # grad_bias: per-block partial sums added with atomics


@pytest.mark.parametrize('s', [1, 4])
def test_tf32x3_mode(s):
    c = {1: 256, 4: 64}[s]
    x, co, mi, wgt, bias, go = _problem(2, c, 8 * s, 8 * s, 8, s, 90 + s, device=DEV)
    want, _, _ = _want(x, co, mi, wgt, bias, go, s, 8)
    with _mode('tf32x3'):
        got, names = _traced(lambda: _raw(x, co, mi, s, wgt, go, 8))
    assert _ran(names, 'coord_cols_kernel<true>', 'DynAggSrc')
    _assert_kernels(names, [], ('PlaneSrc',))
    for name, g, r in zip(('input', 'conv_out', 'weight', 'bias'), got, want):
        e = rel_err(g, r)
        print(f'tf32x3 s={s} grad_{name}: {e:.3g}')
        assert e <= (1.5e-4 if name == 'weight' else max(1e-5, 1.5e-8 * 9 * c)), (name, e)


def _module(c, dg, seed=5):
    torch.manual_seed(seed)
    m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
    m.conv_offset_mask.weight.data.normal_(0, 0.02)
    m.conv_offset_mask.bias.data.normal_(0, 0.3)
    return m


def _module_run(fused, bf16, x, feat0, mi, s, gout, c, dg):
    m = _module(c, dg)
    feat = feat0.clone().requires_grad_(True)
    f_in = feat
    if bf16:
        m.conv_offset_mask.to(memory_format=CL)
        f_in = feat.contiguous(memory_format=CL)
    with torch.autocast('cuda', dtype=torch.bfloat16, enabled=bf16):
        if fused:
            y = m.forward_fused([x, f_in], mi, s, out_slope=0.1, out_like_conv=True)
        else:
            y = m([x, f_in], M.pre_offsets(mi, scales=(s,))[0], out_slope=0.1, out_like_conv=True)
    y.float().backward(gout)
    return (y.float().detach(), feat.grad, m.conv_offset_mask.weight.grad, m.conv_offset_mask.bias.grad, m.weight.grad,
            m.bias.grad)


def test_bf16_channels_last_with_folded_activation():
    """forward_fused(..., out_slope=0.1, out_like_conv=True) under bf16 autocast in channels-last against DynAgg.forward
    (DynAggDCNFunction) on the same map: equal in fp32; in bf16 at least as close to the fp32 result (relative L2).
    The DCN runs in 'tf32x3' so that the fp32 comparison is not dominated by tf32 operand rounding."""
    g = torch.Generator().manual_seed(31)
    b, c, h, w, dg, s = 2, 64, 20, 24, 8, 2
    x = torch.randn(b, c, h, w, generator=g).to(DEV).contiguous(memory_format=CL)
    feat0 = torch.randn(b, c, h, w, generator=g).to(DEV)
    mi = torch.randint(0, (h // s - 2) * (w // s - 2), (b, h // s - 2, w // s - 2), generator=g).to(DEV)
    gout = torch.randn(b, c, h, w, generator=g).to(DEV)
    names = ('y', 'g_feat', 'g_com_w', 'g_com_b', 'g_weight', 'g_bias')
    with _mode('tf32x3'):
        truth = _module_run(False, False, x, feat0, mi, s, gout, c, dg)
        fused32 = _module_run(True, False, x, feat0, mi, s, gout, c, dg)
        two16 = _module_run(False, True, x, feat0, mi, s, gout, c, dg)
        fused16 = _module_run(True, True, x, feat0, mi, s, gout, c, dg)
    for a, r_, name in zip(fused32, truth, names):
        assert rel_err(a, r_) <= 1e-5, (name, rel_err(a, r_))

    def rel_l2(a, r_):
        return float((a.double() - r_.double()).norm() / r_.double().norm().clamp_min(1e-30))
    for a, o, r_, name in zip(fused16, two16, truth, names):
        e_fused, e_two = rel_l2(a, r_), rel_l2(o, r_)
        assert e_fused <= max(1.25 * e_two, 1e-3) and e_fused <= 0.15, (name, e_fused, e_two)


def test_no_grad_forward_fused_is_the_inference_call():
    g = torch.Generator().manual_seed(3)
    b, c, h, w, dg, s = 2, 64, 16, 16, 8, 2
    m = _module(c, dg)
    x = torch.randn(b, c, h, w, generator=g).to(DEV)
    feat = torch.randn(b, c, h, w, generator=g).to(DEV)
    mi = torch.randint(0, 36, (b, 6, 6), generator=g).to(DEV)
    with torch.no_grad():
        y, names = _traced(lambda: m.forward_fused([x, feat], mi, s, out_slope=0.1))
        out = T.conv_bias_to_nchw(feat, m.conv_offset_mask)
        ref, ref_names = _traced(lambda: D.dynagg_dcn_forward(x, out, mi, s, m.weight, m.bias, dg, out_slope=0.1))
    assert torch.equal(y, ref)
    kern = [n for n in names if 'dcn' in n or 'dynagg' in n]
    assert kern and kern == [n for n in ref_names if 'dcn' in n or 'dynagg' in n]
    assert not any('DynAggSrc' in n for n in names)


def test_every_parameter_gets_a_gradient():
    """Before DynAggFusedFunction, forward_fused's output had no grad_fn: DynAgg's weight / bias and the offset
    convolution received no gradient at all."""
    g = torch.Generator().manual_seed(4)
    b, c, h, w, dg, s = 2, 64, 16, 16, 8, 4
    m = _module(c, dg)
    x = torch.randn(b, c, h, w, generator=g).to(DEV).requires_grad_(True)
    feat = torch.randn(b, c, h, w, generator=g).to(DEV)
    mi = torch.randint(0, 4, (b, 2, 2), generator=g).to(DEV)
    y = m.forward_fused([x, feat], mi, s)
    assert y.grad_fn is not None
    y.square().sum().backward()
    for name, p in list(m.named_parameters()) + [('x', x)]:
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()) and bool(p.grad.abs().sum() > 0), name


def test_training_step_on_the_arg_max_map():
    """net_g(lq, max_idx, feats, r) against net_g(lq, pre-offset dict, feats, r): same loss and parameter gradients.
    DCN in 'tf32x3' and convolutions without TF32, so that the comparison sees the DynAgg nodes, not operand rounding.
    The mask logits are held at 0: elsewhere the two sigmoids (__expf / expf) differ in the last bit, that difference
    reaches the next scale's learned offsets, and near initialisation (offsets ~ 0 on integer flows) a point whose
    offset changes sign changes cell -- a one-sided gradient jump, not a defect of either node."""
    from mrefsr_b200.models import MRAPARestorationNet
    g = torch.Generator().manual_seed(8)
    b, r, hr = 2, 2, 64
    h = hr // 4
    lq = torch.rand(b, 3, h, h, generator=g).to(DEV)
    gt = torch.rand(b, 3, hr, hr, generator=g).to(DEV)
    feats = {k: torch.randn(b * r, c, h * s, h * s, generator=g).to(DEV)
             for k, c, s in (('relu3_1', 256, 1), ('relu2_1', 128, 2), ('relu1_1', 64, 4))}
    mi = torch.randint(0, (h - 2) ** 2, (b * r, h - 2, h - 2), generator=g).to(DEV)
    pres = dict(zip(('relu3_1', 'relu2_1', 'relu1_1'), M.pre_offsets(mi)))
    res = []
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with _mode('tf32x3'):
            for src in (pres, mi):
                torch.manual_seed(0)
                net = MRAPARestorationNet(ngf=64, n_blocks=2).to(DEV)
                for name in ('small', 'medium', 'large'):
                    w = getattr(net.dyn_agg_restore, f'{name}_dyn_agg').conv_offset_mask.weight.data
                    w.normal_(0, 1e-3)
                    w[2 * 8 * 9:] = 0       # mask logits exactly 0: both sigmoids give 0.5 (see the docstring)
                loss = torch.nn.functional.l1_loss(net(lq, src, feats, r), gt)
                loss.backward()
                res.append((loss.detach(), {n: p.grad for n, p in net.named_parameters()}))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    assert rel_err(res[1][0], res[0][0]) <= 1e-4
    for n, gr in res[0][1].items():
        assert res[1][1][n] is not None and rel_err(res[1][1][n], gr) <= 1e-4, (n, rel_err(res[1][1][n], gr))


def test_refusals():
    x, co, mi, wgt, bias, go = _problem(1, 64, 16, 16, 8, 2, 1, device=DEV)
    with pytest.raises(RuntimeError, match='fp32'):
        _raw(x, co, mi, 2, wgt, go, 8, mode='fp32')
    x8, co8, mi8, w8, _, go8 = _problem(1, 8, 16, 16, 1, 2, 1, device=DEV)      # C % 32 != 0
    with pytest.raises(RuntimeError, match='needs'):
        _raw(x8, co8, mi8, 2, w8, go8, 1)
    with pytest.raises(RuntimeError):
        _raw(x, co, mi, 2, wgt[:48].contiguous(), go[:, :48].contiguous(), 8)     # Co % 32 != 0
