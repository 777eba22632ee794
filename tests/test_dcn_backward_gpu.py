"""The DCN backward (mrefsr_modulated_deform_conv_backward, csrc/dcn.cu) against the fp64 oracle with the reference's
fp32 sampling positions, on every kernel path the backward selects, at the three training shapes and their chunk
rounds, and at integer and border sampling positions.

Every gradient is compared with rel_err <= TOL.  grad_offset and grad_input are compared a second time on the border
subset -- the sampling points with at least one corner outside the plane, and the input pixels those points touch --
normalised by that subset's own maximum, so that a border bug cannot hide under the interior's larger values.  Each
path case names the kernels it has to reach, checked by name in a torch.profiler trace of the call."""
import pytest
import torch

import mrefsr_b200 as M
import oracle
from mrefsr_b200 import _lib
from mrefsr_b200 import dcn as D
from oracle.dcn import sampling_positions
from tests.util import rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 1e-3   # DCN results within 1e-3 relative error in fp32
NAMES = ('input', 'offset', 'mask', 'weight', 'bias')


def _out_hw(h, w, k, stride, pad, dil):
    return (h + 2 * pad - (dil * (k - 1) + 1)) // stride + 1, (w + 2 * pad - (dil * (k - 1) + 1)) // stride + 1


def _problem(b, c, h, w, co, dg, seed, k=3, stride=1, pad=1, dil=1, groups=1, off_scale=2.0, device='cpu'):
    """(x, offset, mask, weight, bias, grad_output), seeded, on `device`; offsets ~ N(0, off_scale^2)."""
    g = torch.Generator(device=device).manual_seed(seed)
    ho, wo = _out_hw(h, w, k, stride, pad, dil)

    def randn(*shape):
        return torch.randn(*shape, generator=g, device=device)
    x = randn(b, c, h, w)
    off = randn(b, 2 * dg * k * k, ho, wo) * off_scale
    mask = torch.rand(b, dg * k * k, ho, wo, generator=g, device=device)
    wgt = randn(co, c // groups, k, k) * (c // groups * k * k) ** -0.5
    bias = randn(co) * 0.1
    go = randn(b, co, ho, wo)
    return x, off, mask, wgt, bias, go


def _oracle(x, off, mask, wgt, bias, go, k, stride, pad, dil, groups, dg, samples=None):
    """fp64 oracle with fp32 sampling positions, one sample at a time (bounded memory): grad_input / grad_offset /
    grad_mask of `samples` stacked in that order, grad_weight / grad_bias summed over them.  mask None: DCNv1 (its
    grad_mask is None)."""
    samples = range(x.shape[0]) if samples is None else samples
    per, gw, gb = ([], [], []), 0, 0
    for i in samples:
        m = torch.ones(1, dg * k * k, *off.shape[2:]) if mask is None else mask[i:i + 1].cpu()
        r = oracle.modulated_deform_conv_backward_oracle(
            x[i:i + 1].cpu(), off[i:i + 1].cpu(), m, wgt.cpu(), None if bias is None else bias.cpu(), go[i:i + 1].cpu(),
            stride, pad, dil, groups, dg, dtype=torch.float64, fp32_positions=True)
        for lst, t in zip(per, r[:3]):
            lst.append(t)
        gw = gw + r[3]
        gb = gb + r[4] if bias is not None else None
    gi, goff, gm = (torch.cat(t) for t in per)
    return gi, goff, (None if mask is None else gm), gw, gb


def _border_sets(off, h, w, c, k, stride, pad, dil, dg):
    """Boolean masks (over grad_offset, over grad_input) of the sampling points with at least one bilinear corner
    outside the plane, and of the input pixels that such points read (their corners inside the plane)."""
    off = off.detach().cpu().double()
    b, _, ho, wo = off.shape
    kk = k * k
    hy, wx = sampling_positions(off, k, k, (stride,) * 2, (pad,) * 2, (dil,) * 2, dg, torch.float64, fp32_positions=True)
    y0, x0 = torch.floor(hy).long(), torch.floor(wx).long()
    inside = (hy > -1) & (wx > -1) & (hy < h) & (wx < w)
    pts = (y0 < 0) | (y0 + 1 > h - 1) | (x0 < 0) | (x0 + 1 > w - 1)          # [B, dg, K, Ho, Wo]
    off_sel = pts.unsqueeze(3).expand(b, dg, kk, 2, ho, wo).reshape(off.shape)
    touched = torch.zeros(b, dg, h * w, dtype=torch.bool)
    for dy, dx in ((0, 0), (0, 1), (1, 0), (1, 1)):
        yy, xx = y0 + dy, x0 + dx
        ok = pts & inside & (yy >= 0) & (yy <= h - 1) & (xx >= 0) & (xx <= w - 1)
        idx = ok.nonzero()
        touched[idx[:, 0], idx[:, 1], (yy * w + xx)[ok]] = True
    in_sel = touched.view(b, dg, 1, h, w).expand(b, dg, c // dg, h, w).reshape(b, c, h, w)
    return off_sel, in_sel


def _check(got, want, sets=None, what=''):
    """All five gradients within TOL of the oracle; with `sets` (from _border_sets) grad_offset and grad_input also on
    the border subset, normalised by the subset's own maximum."""
    for name, g, r in zip(NAMES, got, want):
        if r is None:
            assert g is None, (what, name)
            continue
        assert g is not None and g.shape == r.shape, (what, name)
        assert rel_err(g, r) <= TOL, (what, name, rel_err(g, r))
    if sets is not None:
        off_sel, in_sel = sets
        for name, g, r, sel in (('offset', got[1], want[1], off_sel), ('input', got[0], want[0], in_sel)):
            if g is None or r is None:
                continue
            assert sel.any(), (what, name, 'empty border subset')
            err = rel_err(g.detach().cpu()[sel], r[sel])
            assert err <= TOL, (what, name + ' (border subset)', err)


def _traced(fn):
    """(fn(), names of the events -- among them the CUDA kernels -- that it ran)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, [e.name for e in prof.events()]


def _assert_kernels(names, reach, avoid, what=''):
    """reach: kernel-name substrings that must run (a (substring, n) pair: exactly n launches); avoid: must not."""
    for k in reach:
        sub, n = k if isinstance(k, tuple) else (k, None)
        cnt = sum(sub in nm for nm in names)
        ran = sorted(set(nm for nm in names if 'dcn' in nm or 'gemm' in nm))
        assert cnt >= 1 if n is None else cnt == n, (what, 'kernel', sub, cnt, ran)
    for sub in avoid:
        assert not any(sub in nm for nm in names), (what, 'unexpected kernel', sub)


def _raw(x, off, mask, wgt, go, k, stride, pad, dil, groups, dg, with_bias=True, **need):
    return D.dcn_backward_raw(x, off, mask, wgt, go, (stride,) * 2, (pad,) * 2, (dil,) * 2, groups, dg, with_bias, **need)


# ---------------------------------------------------------------------------------------------------------------------
# (a) path matrix: each case flips one predicate of the kernel selection in mrefsr_modulated_deform_conv_backward
# ---------------------------------------------------------------------------------------------------------------------
_MERGED = (('gemm_tf32_nt', 2), ('coord_cols', 1), ('bwd_input', 1), ('split_sum', 1), ('gw_permute_add', 1),
           ('bwd_bias', 1))
_NOT_MERGED = ('coord_nhwc', 'bwd_coord_kernel', 'im2col', 'bwd_gcol', 'bwd_weight')

PATH_CASES = {
    # the training step's configuration: 8 / 16 / 32 channels per deform group, merged tcgen05 path
    'production_8ch': dict(p=dict(b=3, c=64, h=40, w=48, co=64, dg=8), reach=_MERGED, avoid=_NOT_MERGED, autograd=True),
    '16ch_per_group': dict(p=dict(b=2, c=128, h=24, w=40, co=128, dg=8), reach=_MERGED, avoid=_NOT_MERGED),
    '32ch_per_group': dict(p=dict(b=2, c=256, h=20, w=20, co=256, dg=8), reach=_MERGED, avoid=_NOT_MERGED),
    # output positions % 4 != 0: no TMA for the grad_weight GEMM -> NHWC coordinate kernel + planar im2col + SIMT GEMM
    'positions_not_mult4': dict(p=dict(b=2, c=64, h=9, w=13, co=64, dg=8),
                                reach=(('gemm_tf32_nt', 1), 'coord_nhwc', 'im2col_kernel', 'bwd_weight', 'bwd_input'),
                                avoid=('coord_cols', 'im2col_planes', 'split_sum', 'bwd_coord_kernel')),
    'no_weight_grad': dict(p=dict(b=2, c=64, h=16, w=16, co=64, dg=8), need=dict(need_weight=False),
                           reach=(('gemm_tf32_nt', 1), 'coord_nhwc', 'bwd_input'),
                           avoid=('im2col', 'bwd_weight', 'split_sum', 'coord_cols', 'gw_permute_add'), v1='input'),
    'no_offset_grad': dict(p=dict(b=2, c=64, h=16, w=16, co=64, dg=8), need=dict(need_offset=False),
                           reach=(('gemm_tf32_nt', 2), 'im2col_planes', 'bwd_input', 'split_sum'),
                           avoid=('coord_cols', 'coord_nhwc', 'bwd_coord_kernel', 'bwd_weight'), v1='parameters'),
    'frozen_input': dict(p=dict(b=2, c=64, h=24, w=20, co=64, dg=8), need=dict(need_input=False),
                         reach=(('gemm_tf32_nt', 2), 'coord_cols', 'split_sum'), avoid=('bwd_input',) + _NOT_MERGED,
                         autograd=True),
    'under_8ch_per_group': dict(p=dict(b=2, c=64, h=16, w=16, co=64, dg=16),
                                reach=(('gemm_tf32_nt', 1), 'bwd_coord_kernel', 'im2col_kernel', 'bwd_weight'),
                                avoid=('coord_cols', 'coord_nhwc', 'im2col_planes')),
    'co_not_mult4': dict(p=dict(b=2, c=64, h=16, w=16, co=30, dg=8),
                         reach=('bwd_gcol', 'coord_cols', ('gemm_tf32_nt', 1), 'split_sum'),
                         avoid=('coord_nhwc', 'im2col', 'bwd_weight')),
    'stride2_dil2': dict(p=dict(b=2, c=64, h=24, w=32, co=64, dg=8, stride=2, pad=2, dil=2), reach=_MERGED,
                         avoid=_NOT_MERGED),
    'kernel5x5': dict(p=dict(b=2, c=64, h=16, w=20, co=64, dg=8, k=5, pad=2), reach=_MERGED, avoid=_NOT_MERGED),
    'kernel5x5_no_weight_grad': dict(p=dict(b=2, c=64, h=16, w=20, co=64, dg=8, k=5, pad=2),
                                     need=dict(need_weight=False), reach=('coord_nhwc',), avoid=('coord_cols', 'im2col')),
    'stride2_no_offset_grad': dict(p=dict(b=2, c=64, h=24, w=32, co=64, dg=8, stride=2, pad=2, dil=2),
                                   need=dict(need_offset=False), reach=('im2col_planes', 'split_sum'),
                                   avoid=('coord_cols', 'coord_nhwc', 'im2col_kernel')),
    # exact-fp32 CUDA-core mode, 48 x 64 = 3072 positions: two 2048-position chunks of the SIMT grad_weight kernel
    'fp32_mode_pchunks': dict(p=dict(b=2, c=16, h=48, w=64, co=16, dg=2), mode='fp32',
                              reach=('bwd_gcol', 'bwd_coord_kernel', 'im2col_kernel', 'bwd_weight', 'bwd_input'),
                              avoid=('gemm_tf32_nt', 'coord_cols', 'coord_nhwc', 'im2col_planes')),
    'fp32_mode_groups2': dict(p=dict(b=2, c=16, h=48, w=64, co=16, dg=2, groups=2), mode='fp32',
                              reach=('bwd_gcol', 'bwd_coord_kernel', 'im2col_kernel', 'bwd_weight'),
                              avoid=('gemm_tf32_nt', 'coord_cols', 'coord_nhwc')),
    # DCNv1 (no mask) on the production shape
    'dcnv1_production': dict(p=dict(b=3, c=64, h=40, w=48, co=64, dg=8), no_mask=True, reach=_MERGED, avoid=_NOT_MERGED),
}


@pytest.mark.parametrize('case', list(PATH_CASES))
def test_backward_paths_vs_oracle(case):
    spec = PATH_CASES[case]
    p = dict(spec['p'])
    b, c, h, w, co, dg = (p.pop(n) for n in ('b', 'c', 'h', 'w', 'co', 'dg'))
    k, stride, pad, dil, groups = p.get('k', 3), p.get('stride', 1), p.get('pad', 1), p.get('dil', 1), p.get('groups', 1)
    need = spec.get('need', {})
    geo = (k, stride, pad, dil, groups, dg)
    x, off, mask, wgt, bias, go = _problem(b, c, h, w, co, dg, 7, **p)
    if spec.get('no_mask'):
        mask = None
    want = list(_oracle(x, off, mask, wgt, bias, go, *geo))
    if not need.get('need_input', True):
        want[0] = None
    if not need.get('need_offset', True):
        want[1] = want[2] = None
    if not need.get('need_weight', True):
        want[3] = None
    sets = _border_sets(off, h, w, c, k, stride, pad, dil, dg)
    xd, od, wd, gd, bd = (t.to(DEV) for t in (x, off, wgt, go, bias))
    md = None if mask is None else mask.to(DEV)
    D.set_default_mode(spec.get('mode', 'auto'))
    try:
        got, names = _traced(lambda: _raw(xd, od, md, wd, gd, *geo, **need))
        _check(got, want, sets, case)
        _assert_kernels(names, spec['reach'], spec['avoid'], case)
        if spec.get('autograd'):
            # the same backward through the autograd Function (frozen input: x does not require grad)
            ts = [t.clone().requires_grad_(True) for t in (od, md, wd, bd)]
            xa = xd.clone().requires_grad_(need.get('need_input', True))
            y = M.modulated_deform_conv(xa, ts[0], ts[1], ts[2], ts[3], stride, pad, dil, groups, dg)
            y.backward(gd)
            _check((xa.grad, ts[0].grad, ts[1].grad, ts[2].grad, ts[3].grad), want, sets, case + ' (autograd)')
    finally:
        D.set_default_mode('auto')
    if spec.get('v1') == 'input':
        # DCNv1 export backward_input: grad_input and grad_offset with an implicit all-ones mask
        want1 = _oracle(x, off, None, wgt, None, go, *geo)
        gi, goff = torch.zeros_like(xd), torch.zeros_like(od)
        names = _traced(lambda: D.ext.deform_conv_backward_input(xd, od, gd, gi, goff, wd, xd.new_empty(0), k, k, stride,
                                                                 stride, pad, pad, dil, dil, groups, dg, 1))[1]
        _check((gi, goff, None, None, None), (want1[0], want1[1], None, None, None), sets, case + ' (DCNv1 export)')
        _assert_kernels(names, ('coord_nhwc', 'bwd_input'), ('im2col', 'bwd_weight'), case + ' (DCNv1 export)')
    if spec.get('v1') == 'parameters':
        # DCNv1 export backward_parameters: grad_weight only, scaled and added to the caller's buffer
        want1 = _oracle(x, off, None, wgt, None, go, *geo)
        gw = torch.full_like(wd, 0.25)
        names = _traced(lambda: D.ext.deform_conv_backward_parameters(xd, od, gd, gw, xd.new_empty(0), xd.new_empty(0), k,
                                                                      k, stride, stride, pad, pad, dil, dil, groups, dg,
                                                                      0.5, 1))[1]
        assert rel_err(gw, 0.25 + 0.5 * want1[3]) <= TOL
        _assert_kernels(names, (('gemm_tf32_nt', 1), 'im2col_planes', 'split_sum'),
                        ('coord_cols', 'coord_nhwc', 'bwd_input', 'bwd_gcol'), case + ' (DCNv1 export)')


# ---------------------------------------------------------------------------------------------------------------------
# (b) chunk rounds at the three training shapes (12 images x 5 references folded would be B = 60)
# ---------------------------------------------------------------------------------------------------------------------
_PER_ROUND_LAUNCHES = 5    # merged path: columns GEMM, coord_cols, bwd_input, grad_weight GEMM, split_sum


@pytest.mark.parametrize('shape', [dict(b=20, c=64, hw=160, nb=18), dict(b=40, c=128, hw=80, nb=36),
                                   dict(b=60, c=256, hw=40, nb=60)], ids=['c64_160', 'c128_80', 'c256_40'])
def test_chunk_rounds_at_training_shapes(shape):
    """The 1 GiB chunk loop at the training shapes (dg 8, 3x3): rounds of 18 + 2 and 36 + 4 samples, and the one-round
    batch-60 call.  grad_output is non-zero on the first / last sample of each round only: those samples against the
    oracle, every other sample's input / offset / mask gradients exactly 0.  Then a dense call against the two
    single-round sub-batch calls: grad_offset / grad_mask bit for bit (plain stores fed by per-sample GEMM tiles),
    grad_input up to atomics order, grad_weight up to the fp32 order of the split-K sums."""
    b, c, hw, nb = (shape[n] for n in ('b', 'c', 'hw', 'nb'))
    dg, geo = 8, (3, 1, 1, 1, 1, 8)
    x, off, mask, wgt, bias, go_dense = _problem(b, c, hw, hw, c, dg, 1000 + c, device=DEV)
    off[:, :, ::7, ::5] *= 8                      # a few large offsets
    picks = [0, nb - 1, nb, b - 1] if nb < b else [0, b // 2, b - 1]
    go = torch.zeros_like(go_dense)
    go[picks] = go_dense[picks]
    n0 = _lib.launch_count()
    got = _raw(x, off, mask, wgt, go, *geo)
    torch.cuda.synchronize()
    n_full = _lib.launch_count() - n0
    others = [i for i in range(b) if i not in picks]
    for name, t in zip(NAMES[:3], got[:3]):
        assert bool((t[others] == 0).all()), (name, 'gradient of a sample whose grad_output is 0')
    want = _oracle(x, off, mask, wgt, bias, go, *geo, samples=picks)
    pk = torch.tensor(picks, device=DEV)
    sets = _border_sets(off[pk], hw, hw, c, *geo[:4], dg)
    _check([t[pk] for t in got[:3]] + list(got[3:]), want, sets, 'sparse grad_output')
    if nb == b:
        return
    # dense grad_output: one two-round call against the two single-round calls on [0:nb] and [nb:b]
    n0 = _lib.launch_count()
    full = _raw(x, off, mask, wgt, go_dense, *geo)
    torch.cuda.synchronize()
    n_dense = _lib.launch_count() - n0
    parts = []
    for lo, hi in ((0, nb), (nb, b)):
        n0 = _lib.launch_count()
        parts.append(_raw(*(t[lo:hi].contiguous() for t in (x, off, mask)), wgt, go_dense[lo:hi].contiguous(), *geo))
        torch.cuda.synchronize()
        n_part = _lib.launch_count() - n0
        assert n_dense - n_part == _PER_ROUND_LAUNCHES and n_full == n_dense, (n_dense, n_part, n_full)
    for i, name in ((1, 'offset'), (2, 'mask')):
        assert torch.equal(full[i][:nb], parts[0][i]) and torch.equal(full[i][nb:], parts[1][i]), name
    gi_parts = torch.cat((parts[0][0], parts[1][0]))
    assert rel_err(full[0], gi_parts) <= 1e-6, rel_err(full[0], gi_parts)
    gw_sum = parts[0][3].double() + parts[1][3].double()
    gb_sum = parts[0][4].double() + parts[1][4].double()
    e_w, e_b = rel_err(full[3], gw_sum), rel_err(full[4], gb_sum)
    print(f'chunked B={b} C={c} {hw}x{hw}: grad_weight vs sum of the two sub-batch calls rel_err {e_w:.3g}, '
          f'grad_bias {e_b:.3g}')
    assert e_w <= 1e-4 and e_b <= 1e-4, (e_w, e_b)


# ---------------------------------------------------------------------------------------------------------------------
# (c) integer and border sampling positions: zero learned offsets plus integer flows, the state of every DynAgg at
# initialisation (DynAgg.init_offset zeroes conv_offset_mask)
# ---------------------------------------------------------------------------------------------------------------------
def _flow_pre_offsets(b, h, w, seed, fractional=False):
    """pre-offsets [B, 9, H, W, 2] (x, y) whose 3x3 sampling points (stride 1, pad 1) land on chosen rows / columns:
    exactly -1, 0, H-1, H and beyond (and the interior) with integer flows; with `fractional`, half the points instead
    sit in (-1, 0) or (H-1, H), where some corners are inside the plane and some are not."""
    g = torch.Generator().manual_seed(seed)

    def axis(n, base):
        edges = torch.tensor([-3., -2., -1., 0., 1., n - 2., n - 1., n, n + 1., n + 2.])
        t = edges[torch.randint(0, len(edges), base.shape, generator=g)]
        t = torch.where(torch.rand(base.shape, generator=g) < 0.3, torch.randint(0, n, base.shape, generator=g).float(), t)
        if fractional:
            u = 0.05 + 0.9 * torch.rand(base.shape, generator=g)
            frac = torch.where(torch.rand(base.shape, generator=g) < 0.5, -1 + u, n - 1 + u)
            t = torch.where(torch.rand(base.shape, generator=g) < 0.5, frac, t)
        return t - base
    k = torch.arange(9)
    by = (torch.arange(h).view(1, 1, h, 1) - 1 + (k // 3).view(1, 9, 1, 1)).float().expand(b, 9, h, w)
    bx = (torch.arange(w).view(1, 1, 1, w) - 1 + (k % 3).view(1, 9, 1, 1)).float().expand(b, 9, h, w)
    return torch.stack((axis(w, bx), axis(h, by)), -1).contiguous()


@pytest.mark.parametrize('kind', ['integer', 'fractional'])
def test_integer_and_border_positions_raw(kind):
    """Offsets = integer flows (+ border fractions): at exact integers both position definitions agree and the offset
    gradient is the reference's one-sided difference.  All gradients within TOL, grad_offset also tap by tap, each tap
    normalised by its own maximum."""
    b, c, h, w, dg = 2, 64, 24, 20, 8
    pre = _flow_pre_offsets(b, h, w, 3 if kind == 'integer' else 4, fractional=kind == 'fractional')
    off, _ = oracle.dynagg_offsets_oracle(torch.zeros(b, 3 * dg * 9, h, w), pre, dg)
    x, _, mask, wgt, bias, go = _problem(b, c, h, w, c, dg, 11)
    geo = (3, 1, 1, 1, 1, dg)
    hy, wx = sampling_positions(off.double(), 3, 3, (1, 1), (1, 1), (1, 1), dg, torch.float64, fp32_positions=True)
    for t, n in ((hy, h), (wx, w)):
        for v in (-1, 0, n - 1, n):
            assert bool((t == v).any()), v                  # the exact edges are sampled
    if kind == 'fractional':
        assert bool(((hy > -1) & (hy < 0)).any()) and bool(((hy > h - 1) & (hy < h)).any())
    want = _oracle(x, off, mask, wgt, bias, go, *geo)
    sets = _border_sets(off, h, w, c, 3, 1, 1, 1, dg)
    got, names = _traced(lambda: _raw(*(t.to(DEV) for t in (x, off, mask, wgt, go)), *geo))
    _assert_kernels(names, _MERGED, _NOT_MERGED)
    _check(got, want, sets, kind)
    gt = got[1].cpu().double().view(b, dg, 9, 2, h, w)
    wt = want[1].view(b, dg, 9, 2, h, w)
    for tap in range(9):
        r = wt[:, :, tap]
        assert float((gt[:, :, tap] - r).abs().max() / r.abs().max()) <= TOL, tap


@pytest.mark.parametrize('fused', [True, False])
def test_dynagg_at_initialisation_vs_oracle(fused):
    """DynAgg.forward in its initial state (conv_offset_mask zeroed: offsets = the integer pre-offsets, masks 0.5),
    as the one autograd node (DynAggDCNFunction) and as the two operator Functions: x / weight / bias gradients against
    the oracle, and the gradients of the offset convolution against fp64 conv2d fed with the oracle's
    [grad_offset, grad_mask * m (1 - m)]."""
    import torch.nn.functional as F
    b, c, h, w, dg = 2, 64, 24, 20, 8
    pre = _flow_pre_offsets(b, h, w, 5)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(b, c, h, w, generator=g)
    feat = torch.randn(b, c, h, w, generator=g)
    go = torch.randn(b, c, h, w, generator=g)
    m = M.DynAgg(c, c, 3, stride=1, padding=1, dilation=1, deform_groups=dg, extra_offset_mask=True).to(DEV)
    assert not m.conv_offset_mask.weight.any() and not m.conv_offset_mask.bias.any()
    m.fused_autograd = fused
    xd = x.to(DEV).requires_grad_(True)
    fd = feat.to(DEV).requires_grad_(True)
    old_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        y = m([xd, fd], pre.to(DEV))
        y.backward(go.to(DEV))
    finally:
        torch.backends.cudnn.allow_tf32 = old_tf32
    off, mask = oracle.dynagg_offsets_oracle(torch.zeros(b, 3 * dg * 9, h, w), pre, dg)
    assert bool((mask == 0.5).all())
    wgt, bias = m.weight.detach().cpu(), m.bias.detach().cpu()
    want = _oracle(x, off, mask, wgt, bias, go, 3, 1, 1, 1, 1, dg)
    sets = _border_sets(off, h, w, c, 3, 1, 1, 1, dg)
    _check((xd.grad, None, None, m.weight.grad, m.bias.grad), (want[0], None, None, want[3], want[4]), sets)
    mk = mask.double()
    g_conv = torch.cat((want[1], want[2] * mk * (1 - mk)), 1)
    f64 = feat.double().requires_grad_(True)
    w64 = torch.zeros(3 * dg * 9, c, 3, 3, dtype=torch.float64, requires_grad=True)
    b64 = torch.zeros(3 * dg * 9, dtype=torch.float64, requires_grad=True)
    F.conv2d(f64, w64, b64, 1, 1).backward(g_conv)
    assert rel_err(fd.grad, f64.grad) <= TOL            # zero weights: 0, like the reference
    assert rel_err(m.conv_offset_mask.weight.grad, w64.grad) <= TOL
    assert rel_err(m.conv_offset_mask.bias.grad, b64.grad) <= TOL


# ---------------------------------------------------------------------------------------------------------------------
# (d) determinism (csrc/dcn.cu: one thread owns a (group, tap, position) of grad_offset / grad_mask; the split-K
# partial sums of grad_weight are added in a fixed order)
# ---------------------------------------------------------------------------------------------------------------------
def test_backward_is_deterministic():
    x, off, mask, wgt, bias, go = (t.to(DEV) for t in _problem(3, 64, 40, 48, 64, 8, 21))
    a = _raw(x, off, mask, wgt, go, 3, 1, 1, 1, 1, 8)
    b = _raw(x, off, mask, wgt, go, 3, 1, 1, 1, 1, 8)
    for i in (1, 2, 3):
        assert torch.equal(a[i], b[i]), NAMES[i]
