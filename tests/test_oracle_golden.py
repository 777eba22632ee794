"""Pin the CPU oracle against vectors produced by the unmodified reference
(tests/golden/make_golden.py).  CPU only."""
import pytest
import torch

import oracle
from oracle.dcn import modulated_deform_conv_c, modulated_deform_conv_backward_c

MATCH_CASES = ['rand', 'shift', 'zeropad', 'raw', 'nonorm', 'strided', 'c256']


@pytest.mark.parametrize('case', MATCH_CASES)
@pytest.mark.parametrize('use_conv', [True, False])
def test_matcher_oracle_matches_reference(golden, case, use_conv):
    g = golden('matcher')
    kw = eval(str(g(f'{case}.kw')))
    idx, val, gap = oracle.feature_match_index_oracle(g(f'{case}.fi'), g(f'{case}.fr'), use_conv=use_conv,
                                                      return_gap=True, **kw)
    ref_idx, ref_val = g(f'{case}.idx'), g(f'{case}.val')
    assert idx.shape == ref_idx.shape and idx.dtype == torch.int64
    # values: 1e-5 abs on O(1) similarities (fp32 summation order differs between conv2d and matmul)
    scale = max(1.0, ref_val.abs().max().item())
    assert (val - ref_val).abs().max().item() <= 1e-5 * scale
    # indices exact wherever the top-2 gap is resolvable (north star: gap >= 1e-5)
    bad = (idx != ref_idx) & (gap >= 1e-5 * scale)
    assert not bad.any()
    if use_conv and case != 'zeropad':
        assert torch.equal(idx, ref_idx)


@pytest.mark.parametrize('case', ['rand', 'zeropad', 'raw', 'strided'])
def test_matcher_oracle_chunked_equals_full(golden, case):
    """The chunked evaluation used at the native validation shapes (125^2 / 128^2 grids) is the same function."""
    g = golden('matcher')
    kw = eval(str(g(f'{case}.kw')))
    full = oracle.feature_match_index_oracle(g(f'{case}.fi'), g(f'{case}.fr'), return_gap=True, dtype=torch.float64, **kw)
    part = oracle.feature_match_index_oracle(g(f'{case}.fi'), g(f'{case}.fr'), return_gap=True, dtype=torch.float64,
                                             chunk=7, **kw)
    assert torch.equal(full[0], part[0])
    assert (full[1] - part[1]).abs().max() < 1e-12 and (full[2] - part[2]).abs().max() < 1e-12


def test_matcher_shift_known_answer(golden):
    g = golden('matcher')
    idx = g('shift.idx')
    hp, wp = idx.shape
    ys, xs = torch.meshgrid(torch.arange(hp), torch.arange(wp), indexing='ij')
    # ref = input shifted by (+3, +2): input patch (y, x) sits at ref (y-3, x-2) when that is inside
    inside = (ys >= 3) & (xs >= 2)
    assert torch.equal(idx[inside], ((ys - 3) * wp + (xs - 2))[inside])
    assert (g('shift.val')[inside] > 0.999).all()


def test_matcher_zero_plateau_first_index(golden):
    g = golden('matcher')
    idx, val = g('zeropad.idx'), g('zeropad.val')
    # input rows >= 12 are zero => all similarities are exactly 0 => first reference index wins
    assert (idx[12:] == 0).all() and (val[12:] == 0).all()
    o_idx, _ = oracle.feature_match_index_oracle(g('zeropad.fi'), g('zeropad.fr'), is_norm=True, norm_input=True)
    assert (o_idx[12:] == 0).all()


def test_sample_patches_layout(golden):
    g = golden('matcher')
    assert torch.equal(oracle.sample_patches_oracle(g('patches.x'), 3, 1), g('patches.y'))


def test_pre_offsets_oracle(golden):
    g = golden('correspondence')
    idx = g('max_idx')
    for b in range(idx.shape[0]):
        pre = oracle.pre_offsets_oracle(idx[b])
        for name in ('relu3_1', 'relu2_1', 'relu1_1'):
            assert torch.equal(pre[name], g(name)[b]), name
    # and the matcher feeding it
    import torch.nn.functional as F
    f1, f2 = g('f1'), g('f2')
    c, h, w = f1.shape[1:]
    for b in range(idx.shape[0]):
        a = F.normalize(f1[b].reshape(c, -1), dim=0).view(c, h, w)
        r = F.normalize(f2[b].reshape(c, -1), dim=0).view(c, h, w)
        oi, _, gap = oracle.feature_match_index_oracle(a, r, is_norm=True, norm_input=True, return_gap=True)
        assert not ((oi != idx[b]) & (gap >= 1e-5)).any()


@pytest.mark.parametrize('case', ['small', 'big_offsets'])
@pytest.mark.parametrize('impl', ['torch', 'c'])
def test_dcn_oracle_forward_backward(golden, case, impl):
    g = golden('dynagg')
    dg = int(g(f'{case}.dg'))
    x, off, mask, w, b = (g(f'{case}.{k}') for k in ('x', 'offset', 'mask', 'weight', 'bias'))
    fwd = oracle.modulated_deform_conv_oracle if impl == 'torch' else modulated_deform_conv_c
    bwd = oracle.modulated_deform_conv_backward_oracle if impl == 'torch' else modulated_deform_conv_backward_c
    y = fwd(x, off, mask, w, b, 1, 1, 1, 1, dg)
    ref = g(f'{case}.y')
    assert (y - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    grads = bwd(x, off, mask, w, b, g(f'{case}.go'), 1, 1, 1, 1, dg)
    for got, key in zip(grads, ('gx', 'goffset', 'gmask', 'gweight', 'gbias')):
        r = g(f'{case}.{key}')
        assert (got - r).abs().max().item() <= 2e-5 * max(1.0, r.abs().max().item()), key


@pytest.mark.parametrize('case', ['small', 'big_offsets'])
def test_dynagg_glue_oracle(golden, case):
    g = golden('dynagg')
    dg = int(g(f'{case}.dg'))
    off, mask = oracle.dynagg_offsets_oracle(g(f'{case}.conv_out'), g(f'{case}.pre'), dg)
    assert torch.equal(off, g(f'{case}.offset'))
    assert torch.allclose(mask, g(f'{case}.mask'), rtol=0, atol=1e-7)


@pytest.mark.parametrize('case', ['t5', 't1', 'pad'])
def test_fusion_oracle(golden, case):
    g = golden('fusion')
    t = int(g(f'{case}.t'))
    out = oracle.mrapa_attention_oracle(g(f'{case}.emb_t'), g(f'{case}.emb'), g(f'{case}.ass'), t)
    ref = g(f'{case}.core_out')
    assert out.shape == ref.shape
    assert (out - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())
    if t == 1:   # single reference: softmax == 1, core is the identity on ass
        assert torch.allclose(out, g(f'{case}.ass'), atol=1e-7)


def test_dcnv1_oracle(golden):
    """DCNv1 = the same sampling rule with an all-ones mask and no bias."""
    g = golden('dcnv1')
    dg, groups = int(g('dg')), int(g('groups'))
    x, off, w = g('x'), g('offset'), g('weight')
    ones = torch.ones(x.shape[0], dg * 9, x.shape[2], x.shape[3])
    y = oracle.modulated_deform_conv_oracle(x, off, ones, w, None, 1, 1, 1, groups, dg)
    assert (y - g('y')).abs().max().item() <= 1e-5 * g('y').abs().max().item()
    gi, goff, _, gw, _ = oracle.modulated_deform_conv_backward_oracle(x, off, ones, w, None, g('go'), 1, 1, 1, groups, dg)
    for got, key in ((gi, 'gx'), (goff, 'goffset'), (gw, 'gweight')):
        assert (got - g(key)).abs().max().item() <= 2e-5 * max(1.0, g(key).abs().max().item()), key


def _flip_problem(seed=0):
    """A DCN problem (offsets ~ N(0, 2^2), dg 2, stride / dilation 1 and 2) in which a few offsets are -2^-25: at a base
    position n >= 1, n - 2^-25 rounds to n in fp32, so those sampling points change cell between the exact and the
    fp32 position."""
    g = torch.Generator().manual_seed(seed)
    b, c, h, w, dg = 2, 8, 9, 11, 2
    x = torch.randn(b, c, h, w, generator=g)
    off = torch.randn(b, 2 * dg * 9, h, w, generator=g) * 2
    mask = torch.rand(b, dg * 9, h, w, generator=g)
    wgt = torch.randn(6, c, 3, 3, generator=g)
    bias = torch.randn(6, generator=g)
    go = torch.randn(b, 6, h, w, generator=g)
    off.view(-1)[torch.randperm(off.numel(), generator=g)[:40]] = -2.0 ** -25
    return x, off, mask, wgt, bias, go, dg


def test_dcn_oracle_fp32_positions_are_the_fp32_sums():
    from oracle.dcn import sampling_positions
    x, off, mask, wgt, bias, go, dg = _flip_problem()
    for stride, pad, dil in ((1, 1, 1), (2, 2, 2)):
        ho = (x.shape[2] + 2 * pad - (2 * dil + 1)) // stride + 1
        wo = (x.shape[3] + 2 * pad - (2 * dil + 1)) // stride + 1
        o = off[:, :, :ho, :wo].contiguous()
        b = o.shape[0]
        him, wim = sampling_positions(o.double(), 3, 3, (stride, stride), (pad, pad), (dil, dil), dg, torch.float64,
                                      fp32_positions=True)
        assert him.dtype == torch.float64 and him.shape == (b, dg, 9, ho, wo)
        ov = o.view(b, dg, 9, 2, ho, wo)
        ys = torch.arange(ho).view(ho, 1) * stride - pad
        xs = torch.arange(wo).view(1, wo) * stride - pad
        for k in range(9):
            by = (ys + (k // 3) * dil).float()
            bx = (xs + (k % 3) * dil).float()
            assert torch.equal(him[:, :, k], (by + ov[:, :, k, 0]).double())       # torch's float32 sum, bit for bit
            assert torch.equal(wim[:, :, k], (bx + ov[:, :, k, 1]).double())
        # exact positions: the fp64 sum; the two differ by at most one fp32 rounding
        ehim, _ = sampling_positions(o.double(), 3, 3, (stride, stride), (pad, pad), (dil, dil), dg, torch.float64)
        assert (ehim - him).abs().max() <= 2.0 ** -24 * ehim.abs().max()
    # straight-through: the derivative with respect to the offset is 1
    o = off.double().requires_grad_(True)
    him, wim = sampling_positions(o, 3, 3, (1, 1), (1, 1), (1, 1), dg, torch.float64, fp32_positions=True)
    (him.sum() + 2 * wim.sum()).backward()
    ov = o.grad.view(o.shape[0], dg, 9, 2, *o.shape[2:])
    assert bool((ov[:, :, :, 0] == 1).all()) and bool((ov[:, :, :, 1] == 2).all())


def test_dcn_oracle_fp32_positions_equal_exact_where_no_point_changes_cell():
    """Both position definitions give the same forward and gradients, except grad_offset at the points whose cell the
    fp32 rounding changes (the bilinear sample is continuous across a cell edge, its derivative is not)."""
    from oracle.dcn import sampling_positions
    x, off, mask, wgt, bias, go, dg = _flip_problem()
    f64 = torch.float64
    h, w = x.shape[2:]
    hx, wx = sampling_positions(off.double(), 3, 3, (1, 1), (1, 1), (1, 1), dg, f64)
    h32, w32 = sampling_positions(off.double(), 3, 3, (1, 1), (1, 1), (1, 1), dg, f64, fp32_positions=True)

    def cell(y, x_):    # the cell a point reads, or -9 when it reads nothing
        inside = (y > -1) & (x_ > -1) & (y < h) & (x_ < w)
        return torch.where(inside, torch.floor(y), -9.0), torch.where(inside, torch.floor(x_), -9.0)
    cy, cx = cell(hx, wx)
    cy32, cx32 = cell(h32, w32)
    flip = (cy != cy32) | (cx != cx32)                                  # [B, dg, 9, H, W]
    assert 5 <= int(flip.sum()) <= 40
    y = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, dg, dtype=f64)
    y32 = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, dg, dtype=f64, fp32_positions=True)
    assert (y - y32).abs().max() <= 1e-6 * y.abs().max()
    ex = oracle.modulated_deform_conv_backward_oracle(x, off, mask, wgt, bias, go, 1, 1, 1, 1, dg, dtype=f64)
    fp = oracle.modulated_deform_conv_backward_oracle(x, off, mask, wgt, bias, go, 1, 1, 1, 1, dg, dtype=f64,
                                                      fp32_positions=True)
    for a, r, name in zip(fp, ex, ('input', 'offset', 'mask', 'weight', 'bias')):
        if name == 'offset':
            keep = ~flip.unsqueeze(3).expand(-1, -1, -1, 2, -1, -1).reshape(a.shape)
            assert (a - r)[keep].abs().max() <= 1e-6 * r.abs().max(), name
            assert (a - r)[~keep].abs().max() >= 1e-2 * r.abs().max(), name      # and the flips do show
        else:
            assert (a - r).abs().max() <= 1e-6 * r.abs().max(), name


@pytest.mark.parametrize('case', ['small', 'big_offsets'])
def test_dcn_oracle_fp32_positions_golden(golden, case):
    """The reference's own gradients, which come from fp32 positions, are matched with the option on too."""
    g = golden('dynagg')
    dg = int(g(f'{case}.dg'))
    x, off, mask, w, b = (g(f'{case}.{k}') for k in ('x', 'offset', 'mask', 'weight', 'bias'))
    y = oracle.modulated_deform_conv_oracle(x, off, mask, w, b, 1, 1, 1, 1, dg, dtype=torch.float64, fp32_positions=True)
    ref = g(f'{case}.y')
    assert (y - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    grads = oracle.modulated_deform_conv_backward_oracle(x, off, mask, w, b, g(f'{case}.go'), 1, 1, 1, 1, dg,
                                                         dtype=torch.float64, fp32_positions=True)
    for got, key in zip(grads, ('gx', 'goffset', 'gmask', 'gweight', 'gbias')):
        r = g(f'{case}.{key}')
        assert (got - r).abs().max().item() <= 2e-5 * max(1.0, r.abs().max().item()), key
