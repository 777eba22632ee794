"""The 3-pass split-tf32 DCN mode ('tf32x3', MREFSR_DCN_TF32X3): tcgen05 kernels whose operands are split into a tf32
hi and a tf32 lo part (hi.hi + hi.lo + lo.hi, fp32 accumulation), against the fp64 oracle with fp32 sampling positions.

The error floor is set by the tensor core's fp32 accumulator, which on the B200 behaves like round-toward-zero: the
error grows linearly with the number of products accumulated into one output (the chain), about 1e-8 per product
(tools/dcn_x3_accum_sim.py emulates it: 4.95e-6 / 1.12e-5 / 2.63e-5 at K = 9 C = 576 / 1152 / 2304, against
4.4e-6 - 5.2e-6 / 9.3e-6 / 1.76e-5 measured on a B200 at 1000 W; a round-to-nearest accumulator would give < 1e-6).
So results are compared with rel_err <= _tol(chain) = max(1e-5, 1.5e-8 * chain), and the forward also with the 'tf32'
mode's error on the same inputs, which it must beat by GAIN (measured: 15x at C = 256, more at smaller C).  The
measured errors are printed (pytest -s) and recorded as test properties."""
import re

import pytest
import torch

import mrefsr_b200 as M
import oracle
from mrefsr_b200 import _lib
from mrefsr_b200 import dcn as D
from tests.test_dcn_backward_gpu import _oracle, _problem, _raw, _traced
from tests.util import rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
TOL = 1e-5      # fp32-grade: the tf32 mode is within 3e-4 on the same inputs
GAIN = 10       # the 3-pass forward's error at least this many times below the tf32 mode's
TOL_GRAD_WEIGHT = 1.5e-4    # grad_weight at the training shapes: split-K chains of up to ~1e4 positions (measured:
                            # 5.8e-5 / 2.8e-5 / 1.2e-5 at C = 64 / 128 / 256 on a B200 at 1000 W)
FULL_MODEL_BOUND = 1e-5     # measured 2.9e-6 on a B200 at 1000 W (7.3e-5 with the DCN in tf32)
NAMES = ('input', 'offset', 'mask', 'weight', 'bias')


class _default_mode:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        D.set_default_mode(self.mode)

    def __exit__(self, *exc):
        D.set_default_mode('auto')


def _tol(chain):
    """Bound for a result accumulated from `chain` products per output (see the module docstring)."""
    return max(TOL, 1.5e-8 * chain)


def _report(record_property, what, err):
    record_property(what, err)
    print(f'{what}: rel_err {err:.3g}')


def _tf32_split(t):
    """(hi, lo): hi = t rounded to tf32 (low 13 bits cleared), lo = the remainder rounded to tf32, as the kernels do."""
    def rnd(v):
        return ((v.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)
    hi = rnd(t)
    return hi, rnd(t - hi)


# ---------------------------------------------------------------------------------------------------------------------
# forward
# ---------------------------------------------------------------------------------------------------------------------
def _forward_pair(x, off, mask, wgt, bias, dg, stride=1, pad=1, dil=1):
    args = ((stride,) * 2, (pad,) * 2, (dil,) * 2, 1, dg)
    dev = [t.to(DEV) if t is not None else None for t in (x, off, mask, wgt, bias)]
    return (D.dcn_forward_raw(*dev, *args, mode='tf32x3'), D.dcn_forward_raw(*dev, *args, mode='tf32'))


@pytest.mark.parametrize('cfg', [
    dict(b=2, c=64, h=20, w=24, co=64, dg=8),                        # 8 channels per deform group: 2 groups per slab
    dict(b=1, c=128, h=16, w=16, co=128, dg=8),                      # 16: one group per slab
    dict(b=1, c=256, h=10, w=12, co=256, dg=8),                      # 32: a slab inside a group
    dict(b=3, c=32, h=7, w=5, co=96, dg=2, off_scale=5.0),
    dict(b=1, c=64, h=9, w=9, co=32, dg=1, stride=2, pad=1, dil=1),
    dict(b=1, c=64, h=11, w=13, co=64, dg=4, stride=1, pad=2, dil=2),
])
@pytest.mark.parametrize('with_bias', [True, False])
def test_forward_vs_oracle(cfg, with_bias, record_property):
    cfg = dict(cfg)
    b, c, h, w, co, dg = (cfg.pop(k) for k in ('b', 'c', 'h', 'w', 'co', 'dg'))
    stride, pad, dil = cfg.pop('stride', 1), cfg.pop('pad', 1), cfg.pop('dil', 1)
    x, off, mask, wgt, bias, _ = _problem(b, c, h, w, co, dg, 5, stride=stride, pad=pad, dil=dil, **cfg)
    bias = bias if with_bias else None
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, stride, pad, dil, 1, dg, dtype=torch.float64,
                                              fp32_positions=True)
    y3, y1 = _forward_pair(x, off, mask, wgt, bias, dg, stride, pad, dil)
    e3, e1 = rel_err(y3, ref), rel_err(y1, ref)
    _report(record_property, 'x3', e3)
    _report(record_property, 'tf32', e1)
    assert e3 <= _tol(9 * c) and e3 * GAIN <= e1, (e3, e1)


def _flow_case(b, c, h, w, s, flow, seed=31, dg=8):
    """(x, conv_out, max_idx, weight, bias, offset, mask): the flows of test_dcn_gpu's coherent / border test."""
    g = torch.Generator().manual_seed(seed)
    hp, wp = h // s - 2, w // s - 2
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
        elif flow == 'border':
            dy, dx = (hp - 2, wp - 2) if i % 2 == 0 else (-(hp - 2), -(wp - 2))
            m = (ys + dy).clamp(0, hp - 1) * wp + (xs + dx).clamp(0, wp - 1)
        else:                                  # half translation, half random (test_native_grids_vs_oracle)
            coherent = (ys + 3).clamp(0, hp - 1) * wp + (xs - 2).clamp(0, wp - 1)
            m = torch.where(xs < wp // 2, coherent, torch.randint(0, hp * wp, (hp, wp), generator=g))
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
    return x, conv_out, max_idx, wgt, bias, off.float(), mask.float()


@pytest.mark.parametrize('cfg', [dict(b=3, c=64, h=48, w=64, s=4), dict(b=2, c=128, h=40, w=48, s=2),
                                 dict(b=2, c=256, h=24, w=40, s=1), dict(b=2, c=64, h=75, w=75, s=1)])
@pytest.mark.parametrize('flow', ['translate', 'piecewise', 'border'])
def test_coherent_and_border_flows_vs_oracle(cfg, flow, record_property):
    """Fused DynAgg and the operator entry point in the 3-pass mode on the coherent / border flows; the 75 x 75 grid
    takes the linear row mapping of the CTA tiles, the others square patches."""
    b, c, h, w, s = (cfg[k] for k in ('b', 'c', 'h', 'w', 's'))
    x, conv_out, max_idx, wgt, bias, off, mask = _flow_case(b, c, h, w, s, flow)
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, 8, dtype=torch.float64,
                                              fp32_positions=True)
    with _default_mode('tf32x3'):
        y_fused = D.dynagg_dcn_forward(x.to(DEV), conv_out.to(DEV), max_idx.to(DEV), s, wgt.to(DEV), bias.to(DEV), 8)
    y3, y1 = _forward_pair(x, off, mask, wgt, bias, 8)
    e_f, e3, e1 = rel_err(y_fused, ref), rel_err(y3, ref), rel_err(y1, ref)
    for what, e in (('fused x3', e_f), ('operator x3', e3), ('operator tf32', e1)):
        _report(record_property, what, e)
    assert e_f <= _tol(9 * c) and e3 <= _tol(9 * c) and e3 * GAIN <= e1, (e_f, e3, e1)


@pytest.mark.parametrize('cfg', [dict(c=64, hw=160, s=4), dict(c=128, hw=150, s=2), dict(c=256, hw=75, s=1)])
def test_native_grids_vs_oracle(cfg, record_property):
    """The config-2 / config-3 feature grids (160^2, 150^2, 75^2), fused and operator path."""
    c, hw, s = (cfg[k] for k in ('c', 'hw', 's'))
    x, conv_out, max_idx, wgt, bias, off, mask = _flow_case(1, c, hw, hw, s, 'mixed', seed=hw + c)
    ref = oracle.modulated_deform_conv_oracle(x, off, mask, wgt, bias, 1, 1, 1, 1, 8, dtype=torch.float64,
                                              fp32_positions=True)
    with _default_mode('tf32x3'):
        y_fused = D.dynagg_dcn_forward(x.to(DEV), conv_out.to(DEV), max_idx.to(DEV), s, wgt.to(DEV), bias.to(DEV), 8)
    y3, y1 = _forward_pair(x, off, mask, wgt, bias, 8)
    e_f, e3, e1 = rel_err(y_fused, ref), rel_err(y3, ref), rel_err(y1, ref)
    for what, e in (('fused x3', e_f), ('operator x3', e3), ('operator tf32', e1)):
        _report(record_property, what, e)
    assert e_f <= _tol(9 * c) and e3 <= _tol(9 * c) and e3 * GAIN <= e1, (e_f, e3, e1)


@pytest.mark.parametrize('in_cl', [False, True])
@pytest.mark.parametrize('out_cl', [False, True])
@pytest.mark.parametrize('packed', [False, True])
def test_fused_dynagg_layouts_and_packing(in_cl, out_cl, packed, record_property):
    """Fused DynAgg in the 3-pass mode with NCHW / NHWC input and output and with weights packed once
    (pack_weight(w, 'tf32x3')) against the fp32 operator path on the materialised offsets / masks.  Packed and
    unpacked weights give the same bits; a tf32 packing is refused while the mode is tf32x3."""
    b, c, h, w, s, dg = 2, 64, 32, 40, 2, 8
    x, conv_out, max_idx, wgt, bias, off, mask = _flow_case(b, c, h, w, s, 'piecewise', seed=7)
    xd, cd, md, wd, bd = (t.to(DEV) for t in (x, conv_out, max_idx, wgt, bias))
    ref = D.dcn_forward_raw(xd, off.to(DEV), mask.to(DEV), wd, bd, (1, 1), (1, 1), (1, 1), 1, dg, mode='fp32')
    xin = xd.contiguous(memory_format=torch.channels_last) if in_cl else xd
    with _default_mode('tf32x3'):
        wp = D.pack_weight(wd) if packed else None
        y = D.dynagg_dcn_forward(xin, cd, md, s, wd, bd, dg, out_channels_last=out_cl, weight_packed=wp)
        assert y.is_contiguous(memory_format=torch.channels_last) == out_cl
        if packed:
            assert wp.shape == (c, 2 * 9 * c)
            assert torch.equal(y, D.dynagg_dcn_forward(xin, cd, md, s, wd, bd, dg, out_channels_last=out_cl))
            with pytest.raises(RuntimeError):
                D.dynagg_dcn_forward(xin, cd, md, s, wd, bd, dg, weight_packed=D.pack_weight(wd, 'tf32'))
    e = rel_err(y, ref)
    _report(record_property, 'fused x3 vs fp32 operator', e)
    assert e <= _tol(9 * c), e


def test_fused_dynagg_into_buffers_matches_the_single_output():
    """dynagg_dcn_forward_into (several buffers, and pixel slabs) follows the mode too: same bits as the one-output
    entry point in the 3-pass mode."""
    b, c, h, w, s, dg = 2, 64, 24, 24, 2, 8
    x, conv_out, max_idx, wgt, bias, _, _ = _flow_case(b, c, h, w, s, 'translate', seed=11)
    xd, cd, md, wd, bd = (t.to(DEV) for t in (x, conv_out, max_idx, wgt, bias))
    with _default_mode('tf32x3'):
        y = D.dynagg_dcn_forward(xd, cd, md, s, wd, bd, dg)
        bufs = [torch.full((b, c, h, w), float('nan'), device=DEV) for _ in range(2)]
        D.dynagg_dcn_forward_into(xd, cd, md, s, wd, bd, dg, [t.data_ptr() for t in bufs], 0, 0, 0)
        slabs = [torch.full((b, c, h // 2, w), float('nan'), device=DEV) for _ in range(2)]
        D.dynagg_dcn_forward_into(xd, cd, md, s, wd, bd, dg, [t.data_ptr() for t in slabs], 0, 0, 0, slab_rows=h // 2)
    torch.cuda.synchronize()
    assert torch.equal(bufs[0], y) and torch.equal(bufs[1], y)
    assert torch.equal(torch.cat(slabs, 2), y)
    with _default_mode('tf32'):
        assert not torch.equal(D.dynagg_dcn_forward(xd, cd, md, s, wd, bd, dg), y)


# ---------------------------------------------------------------------------------------------------------------------
# backward
# ---------------------------------------------------------------------------------------------------------------------
def _check_grads(got, want, record_property, what, names=NAMES, tol_weight=TOL):
    for name, g, r in zip(names, got, want):
        e = rel_err(g, r)
        _report(record_property, f'{what} grad_{name}', e)
        assert e <= (tol_weight if name == 'weight' else TOL), (what, name, e)


@pytest.mark.parametrize('shape', [dict(b=20, c=64, hw=160, nb=12), dict(b=40, c=128, hw=80, nb=24),
                                   dict(b=60, c=256, hw=40, nb=48)], ids=['c64_160', 'c128_80', 'c256_40'])
def test_backward_at_training_shapes(shape, record_property):
    """All five gradients at the training shapes (dg 8, 3x3) in the 3-pass mode, which runs them in rounds of 12 + 8,
    24 + 16 and 48 + 12 samples.  grad_output is non-zero on the first / last sample of each round only: those samples
    against the oracle, every other sample's input / offset / mask gradients exactly 0.  The trace shows the 3-pass
    GEMM twice per round and the one-pass GEMM never."""
    b, c, hw, nb = (shape[n] for n in ('b', 'c', 'hw', 'nb'))
    dg, geo = 8, (3, 1, 1, 1, 1, 8)
    x, off, mask, wgt, bias, go_dense = _problem(b, c, hw, hw, c, dg, 2000 + c, device=DEV)
    off[:, :, ::7, ::5] *= 8
    picks = [0, nb - 1, nb, b - 1]
    go = torch.zeros_like(go_dense)
    go[picks] = go_dense[picks]
    with _default_mode('tf32x3'):
        got, names = _traced(lambda: _raw(x, off, mask, wgt, go, *geo))
    gemms = [re.search(r'gemm_tf32_nt_kernel<(\w+)>', n).group(1) for n in names if 'gemm_tf32_nt_kernel' in n]
    assert gemms == ['true'] * 4, gemms
    assert any('dcn_bwd_coord_cols_kernel<true>' in n for n in names)
    others = [i for i in range(b) if i not in picks]
    for name, t in zip(NAMES[:3], got[:3]):
        assert bool((t[others] == 0).all()), (name, 'gradient of a sample whose grad_output is 0')
    want = _oracle(x, off, mask, wgt, bias, go, *geo, samples=picks)
    pk = torch.tensor(picks, device=DEV)
    _check_grads([t[pk] for t in got[:3]] + list(got[3:]), want, record_property, f'B{b} C{c} {hw}^2',
                 tol_weight=TOL_GRAD_WEIGHT)


@pytest.mark.parametrize('case', ['merged', 'weight_only', 'offset_only'])
def test_backward_paths(case, record_property):
    """The 3-pass backward on its other producer paths at a small shape: the column planes written by
    dcn_im2col_planes_kernel (no offset gradient), and no grad_weight GEMM at all (no weight gradient)."""
    need = dict(merged={}, weight_only=dict(need_offset=False, need_input=False),
                offset_only=dict(need_weight=False))[case]
    b, c, h, w, co, dg = 3, 64, 18, 20, 96, 4
    geo = (3, 1, 1, 1, 1, dg)
    x, off, mask, wgt, bias, go = _problem(b, c, h, w, co, dg, 77, device=DEV)
    with _default_mode('tf32x3'):
        got, names = _traced(lambda: _raw(x, off, mask, wgt, go, *geo, **need))
    want = list(_oracle(x, off, mask, wgt, bias, go, *geo))
    if 'need_offset' in need:
        want[1] = want[2] = None
        assert any('dcn_im2col_planes_kernel<true>' in n for n in names)
    if 'need_input' in need:
        want[0] = None
    if 'need_weight' in need:
        want[3] = None
    assert not any('<false>' in n for n in names if 'gemm_tf32_nt_kernel' in n)
    pairs = [(g, r, n) for g, r, n in zip(got, want, NAMES) if r is not None]
    _check_grads([p[0] for p in pairs], [p[1] for p in pairs], record_property, case, names=[p[2] for p in pairs])
    assert all(got[i] is None for i in range(4) if want[i] is None)


@pytest.mark.parametrize('shape', [dict(M=576, N=1600, K=64, batch=3), dict(M=130, N=70, K=36, batch=2),
                                   dict(M=2304, N=6400, K=256, batch=1),
                                   dict(M=64, N=576, K=25600, batch=2, reduce=True, splits=30),
                                   dict(M=96, N=200, K=100, batch=3, reduce=True, splits=7)])
def test_gemm_entry_vs_fp64(shape, record_property):
    """mrefsr_gemm_tf32x3_nt against torch fp64 on the same fp32 operands, at ragged M / N / K, with a shared A and in
    the split-K reduce mode."""
    M_, N_, K_, batch = (shape[k] for k in ('M', 'N', 'K', 'batch'))
    reduce, splits = shape.get('reduce', False), shape.get('splits', 1)
    g = torch.Generator().manual_seed(M_ + N_)
    lda = (K_ + 3) // 4 * 4 + 4
    a = torch.randn(batch if reduce else 1, M_, lda, generator=g).to(DEV)
    b = torch.randn(batch, N_, lda, generator=g).to(DEV)
    (a_hi, a_lo), (b_hi, b_lo) = _tf32_split(a), _tf32_split(b)
    n_out = splits if reduce else batch
    ldd = N_ + 3
    d = torch.full((n_out, M_, ldd), float('nan'), device=DEV)
    p = _lib.ptr
    rc = _lib.lib().mrefsr_gemm_tf32x3_nt(p(a_hi), p(a_lo), lda, M_ * lda if reduce else 0, p(b_hi), p(b_lo), lda,
                                          N_ * lda, p(d), ldd, M_ * ldd, M_, N_, K_, batch, int(reduce), splits,
                                          _lib.stream_ptr(a.device))
    _lib.check(rc, 'mrefsr_gemm_tf32x3_nt')
    torch.cuda.synchronize()
    a64, b64 = a[..., :K_].double().cpu(), b[..., :K_].double().cpu()
    assert torch.isnan(d[..., N_:]).all()
    if reduce:
        ref, out = torch.einsum('zmk,znk->mn', a64, b64), d[..., :N_].double().cpu().sum(0)
    else:
        ref, out = torch.einsum('mk,znk->zmn', a64[0], b64), d[..., :N_].double().cpu()
    e = float((out - ref).abs().max() / ref.abs().max())
    _report(record_property, 'gemm x3', e)
    assert e <= _tol(K_ * batch // splits if reduce else K_), e


# ---------------------------------------------------------------------------------------------------------------------
# kernel choice, refusals, the whole model
# ---------------------------------------------------------------------------------------------------------------------
def test_x3_instantiations_run_in_x3_mode_only():
    """A profiler trace names the 3-pass instantiations (dcn_tc_split_kernel<..., true>, gemm_tf32_nt_kernel<true>, the
    split producers) in the tf32x3 mode, and never in the default mode."""
    x, off, mask, wgt, bias, go = _problem(2, 64, 16, 16, 64, 8, 3, device=DEV)
    ts = [t.clone().requires_grad_(True) for t in (x, off, mask, wgt, bias)]

    def step():
        y = M.modulated_deform_conv(*ts, 1, 1, 1, 1, 8)
        y.backward(go)
        return y
    for mode, x3 in (('tf32x3', True), ('auto', False)):
        with _default_mode(mode):
            _, names = _traced(step)
        fwd = [re.search(r'dcn_tc_split_kernel<(\w+), (\d+), (\w+)>', n).groups() for n in names
               if 'dcn_tc_split_kernel' in n]
        gemm = [re.search(r'gemm_tf32_nt_kernel<(\w+)>', n).group(1) for n in names if 'gemm_tf32_nt_kernel' in n]
        flag = 'true' if x3 else 'false'
        assert fwd and all(f[2] == flag for f in fwd), (mode, fwd)
        assert gemm and all(f == flag for f in gemm), (mode, gemm)
        assert any(f'dcn_bwd_coord_cols_kernel<{flag}>' in n for n in names), mode
        assert any('nchw_to_nhwc_kernel<true, true>' in n for n in names) == x3, mode
        assert any('dcn_weight_repack_x3_kernel' in n for n in names) == x3, mode


@pytest.mark.parametrize('shape', [(1, 8, 6, 6, 8, 2), (1, 48, 6, 6, 32, 1), (1, 64, 6, 6, 48, 8), (1, 64, 6, 6, 64, 16)])
def test_x3_mode_rejects_ineligible(shape):
    """Shapes the tcgen05 kernels cannot take raise in the 3-pass mode, as in the tf32 mode (no silent fp32 path)."""
    b, c, h, w, co, dg = shape
    x, off, mask, wgt, bias, _ = _problem(b, c, h, w, co, dg, 1, device=DEV)
    for mode in ('tf32', 'tf32x3'):
        with pytest.raises(RuntimeError):
            D.dcn_forward_raw(x, off, mask, wgt, bias, (1, 1), (1, 1), (1, 1), 1, dg, mode=mode)


def test_full_model_error_drops_with_x3(golden, record_property):
    """The full_model golden with cuDNN in exact fp32: the SR error with the DCN in the 3-pass mode is smaller than with
    the DCN in tf32, and within FULL_MODEL_BOUND."""
    from mrefsr_b200.models import MRefSRPipeline
    from tests.util import refill_parameters
    m = MRefSRPipeline().eval()
    refill_parameters(m.net_extractor, 1)
    refill_parameters(m.net_map, 2)
    refill_parameters(m.net_g, 3)
    m = m.to(DEV)
    g = golden('full_model')
    lq, up, refs, sr_ref = (g(k).to(DEV) for k in ('lq', 'up', 'refs', 'sr'))
    base = torch.nn.functional.interpolate(lq, None, 4, 'bilinear', False).double().cpu()
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    errs = {}
    try:
        for mode in ('tf32', 'tf32x3'):
            with _default_mode(mode), torch.no_grad():
                sr = m(lq, up, refs).double().cpu()
            errs[mode] = float((sr - sr_ref.double().cpu()).norm() / (sr_ref.double().cpu() - base).norm())
            _report(record_property, f'full model, DCN {mode}', errs[mode])
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert errs['tf32x3'] < errs['tf32'], errs
    assert errs['tf32x3'] <= FULL_MODEL_BOUND, errs
