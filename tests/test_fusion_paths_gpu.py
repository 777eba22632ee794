"""The fusion head's kernels (csrc/fusion.cu and the training epilogue of csrc/trunk.cu) against fp64 references, on
every instantiation their entry points dispatch to, at the model's shapes and at the edges where the kernels branch:
partly empty CTAs, channel counts below the 8 warps of a CTA, misaligned views, more than 8 references, saturated and
tied softmax logits, several rounds of a grid-stride loop and more partial rows than the 32 lanes of the bias-gradient
reduction.

The attention reference is oracle.mrapa_attention_oracle in float64 (its gradients through torch autograd in float64);
the epilogue's reference is a torch float64 expression.  Each case that claims a kernel path checks, by name in a
torch.profiler trace, which instantiations ran."""
import copy
import re

import pytest
import torch
import torch.nn.functional as F

import mrefsr_b200 as M
import oracle
from mrefsr_b200 import fusion as FU
from mrefsr_b200 import trunk as T
from tests.util import rel_err

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
OUT_TOL, GRAD_TOL = 1e-5, 1e-4      # fp32 kernels: output, gradients (rel_err against fp64)
BF16_TOL = 4e-3                     # bf16 I/O: one bf16 rounding of the output plus fp32 accumulation
BF16_TRAIN_TOL = 8e-3               # bf16 channels-last training path: bf16 outputs and gradients


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL = re.compile(r'(mrapa_\w+|bias_act_train_\w+|bias_grad_sum_kernel)(<[^>(]*>)?')


def _norm(name):
    return name.replace('(int)', '').replace(' ', '')


def _traced(fn):
    """(fn(), set of the fusion / training-epilogue kernels it ran, as 'name<template args>' without spaces).
    fn must be repeatable: a trace that holds no device activity at all lost it (seen once in a few hundred traces of
    one session) and is taken again."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            res = fn()
            torch.cuda.synchronize()
        events = prof.events()
        if any(e.device_type == DeviceType.CUDA for e in events):
            break
    ran = set()
    for e in events:
        m = _KERNEL.search(_norm(e.name))
        if m:
            ran.add(m.group(0))
    return res, ran


def _mrapa(ran):
    return {k for k in ran if k.startswith('mrapa_')}


def _expect(*names):
    return {_norm(n) for n in names}


def _randn(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g, device=DEV) * scale


def _core_problem(n, t, c, cv, h, w, seed):
    """q (logits of order 1 at any C), k, v, grad_out: fp32 NCHW on the GPU."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    q = _randn(g, n, c, h, w, scale=1.5 / c ** 0.5)
    k = _randn(g, n * t, c, h, w)
    v = _randn(g, n * t, cv, h, w)
    go = _randn(g, n, cv, h, w)
    return q, k, v, go


def _misaligned(x):
    """A copy of x that is a view one element into its storage: not 16-byte aligned (fp32), not 8-byte aligned (bf16)."""
    y = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)[1:].view(x.shape)
    y.copy_(x)
    assert y.data_ptr() % 8 != 0
    return y


def _oracle_fwd_bwd(q, k, v, go, t):
    """fp64 output and gradients (emb_t, emb, ass) of the attention core."""
    r = [x.detach().double().requires_grad_(True) for x in (q, k, v)]
    out = oracle.mrapa_attention_oracle(r[0], r[1], r[2], t, dtype=torch.float64)
    out.backward(go.double())
    return out.detach(), [x.grad for x in r]


def _run_core(q, k, v, go, t):
    """The public entry under autograd: (output, gradients, kernels run)."""
    leaves = [x.detach().requires_grad_(True) for x in (q, k, v)]   # detach keeps a view's storage offset

    def run():
        out = M.mrapa_attention(leaves[0], leaves[1], leaves[2], t)
        return out.detach(), torch.autograd.grad(out, leaves, go)
    (out, grads), ran = _traced(run)
    return out, grads, ran


def _check_core(q, k, v, go, t, kernels, what=''):
    out, grads, ran = _run_core(q, k, v, go, t)
    assert _mrapa(ran) == _expect(*kernels), (what, sorted(ran))
    ref, rgrads = _oracle_fwd_bwd(q, k, v, go, t)
    assert rel_err(out, ref) <= OUT_TOL, (what, 'out', rel_err(out, ref))
    for a, b, name in zip(grads, rgrads, ('emb_t', 'emb', 'ass')):
        assert torch.isfinite(a).all(), (what, name)
        assert rel_err(a, b) <= GRAD_TOL, (what, name, rel_err(a, b))
    return out, grads


# ---------------------------------------------------------------------------------------------------------------------
# 1. NCHW core, fp32, forward + backward on every instantiation
# ---------------------------------------------------------------------------------------------------------------------
# (n, t, C, Cv, h, w): n >= 2 everywhere (per-image offsets of q / k / v / prob / out / gradients); h*w % 4 == 0 but rarely
# a multiple of the 128 pixels of a CTA (a partly empty last CTA); C or Cv < 8 or not a multiple of 8 (warps without
# channels, uneven slices).
VEC4_SHAPES = {
    1: (2, 1, 32, 64, 12, 20),
    2: (2, 2, 16, 32, 9, 12),
    3: (2, 3, 5, 6, 8, 12),
    4: (2, 4, 64, 128, 16, 20),
    5: (2, 5, 3, 7, 10, 10),
    6: (2, 6, 48, 96, 12, 12),
    7: (2, 7, 24, 40, 20, 20),
    8: (3, 8, 8, 16, 4, 9),
}


@pytest.mark.parametrize('t', sorted(VEC4_SHAPES))
def test_core_vec4_every_reference_count(t):
    n, _, c, cv, h, w = VEC4_SHAPES[t]
    q, k, v, go = _core_problem(n, t, c, cv, h, w, seed=t)
    _check_core(q, k, v, go, t, (f'mrapa_fwd_vec4_kernel<{t}, float>', f'mrapa_bwd_vec4_kernel<{t}>'))


@pytest.mark.parametrize('c,h', [(64, 160), (128, 80), (256, 40)])
def test_core_vec4_training_shapes(c, h):
    """The training step's three scales: t = 5, Cv = 2C, 160^2 / 80^2 / 40^2."""
    q, k, v, go = _core_problem(2, 5, c, 2 * c, h, h, seed=c)
    _check_core(q, k, v, go, 5, ('mrapa_fwd_vec4_kernel<5, float>', 'mrapa_bwd_vec4_kernel<5>'))


def test_core_scalar8_odd_grid():
    """h*w % 4 != 0: the one-pixel-per-lane kernels with TMAX = 8."""
    q, k, v, go = _core_problem(2, 5, 20, 40, 7, 9, seed=21)
    _check_core(q, k, v, go, 5, ('mrapa_fwd_kernel<8>', 'mrapa_bwd_kernel<8>'))


@pytest.mark.parametrize('which', ['emb_t', 'emb', 'ass', 'grad_out'])
def test_core_scalar8_misaligned_view(which):
    """h*w % 4 == 0 and t <= 8, but one tensor is a view that is not 16-byte aligned: the public entry must route the
    kernels that read it to the scalar versions (a misaligned grad_out only concerns the backward)."""
    q, k, v, go = _core_problem(2, 6, 24, 48, 8, 12, seed=22)
    xs = dict(emb_t=q, emb=k, ass=v, grad_out=go)
    xs[which] = _misaligned(xs[which])
    fwd = 'mrapa_fwd_vec4_kernel<6, float>' if which == 'grad_out' else 'mrapa_fwd_kernel<8>'
    _check_core(xs['emb_t'], xs['emb'], xs['ass'], xs['grad_out'], 6, (fwd, 'mrapa_bwd_kernel<8>'), which)


@pytest.mark.parametrize('shape', [(2, 9, 24, 40, 9, 11), (2, 12, 16, 32, 7, 13), (2, 16, 40, 80, 10, 10)])
def test_core_scalar16(shape):
    """9..16 references (TMAX = 16) on grids with h*w % 32 != 0 (a partly empty last CTA)."""
    n, t, c, cv, h, w = shape
    q, k, v, go = _core_problem(n, t, c, cv, h, w, seed=t)
    _check_core(q, k, v, go, t, ('mrapa_fwd_kernel<16>', 'mrapa_bwd_kernel<16>'))


# ---------------------------------------------------------------------------------------------------------------------
# 2. softmax edges: saturated and tied logits, on the vec4 and both scalar forwards
# ---------------------------------------------------------------------------------------------------------------------
EDGE_PATHS = {   # name: (n, t, C, Cv, h, w), kernels
    'vec4': ((2, 5, 16, 32, 8, 12), ('mrapa_fwd_vec4_kernel<5, float>', 'mrapa_bwd_vec4_kernel<5>')),
    'scalar8': ((2, 5, 16, 32, 7, 9), ('mrapa_fwd_kernel<8>', 'mrapa_bwd_kernel<8>')),
    'scalar16': ((2, 12, 16, 32, 6, 11), ('mrapa_fwd_kernel<16>', 'mrapa_bwd_kernel<16>')),
}


@pytest.mark.parametrize('path', list(EDGE_PATHS))
@pytest.mark.parametrize('kind', ['saturated', 'tied'])
def test_softmax_edges(kind, path):
    """Every other pixel is an edge pixel; the rest keep ordinary logits, so that the gradients have a scale to be
    compared at.  saturated: reference w = (p // 2) % t has logit +200, reference w + 1 has -200, the others are of order 1
    (a gap of ~200: exp of the unshifted logit overflows fp32), so the output is reference w's value map.  tied: all
    references have the key of reference 0, so the output is the mean of the value maps."""
    (n, t, c, cv, h, w), kernels = EDGE_PATHS[path]
    q, k, v, go = _core_problem(n, t, c, cv, h, w, seed=31)
    hw = h * w
    p = torch.arange(hw, device=DEV)
    edge = p % 2 == 0
    win = (p // 2) % t
    kk, qq = k.view(n, t, c, hw), q.view(n, c, hw)
    if kind == 'saturated':
        aligned = qq * (200.0 / qq.square().sum(1, keepdim=True))          # <q, aligned> = 200
        for i in range(t):
            lose = edge & ((win + 1) % t == i)
            kk[:, i][:, :, lose] = -aligned[:, :, lose]
            hit = edge & (win == i)
            kk[:, i][:, :, hit] = aligned[:, :, hit]
    else:
        for i in range(1, t):
            kk[:, i][:, :, edge] = kk[:, 0][:, :, edge]
    out, _ = _check_core(q, k, v, go, t, kernels, f'{kind}/{path}')
    vv = v.view(n, t, cv, hw)
    if kind == 'saturated':
        want = vv.gather(1, win.view(1, 1, 1, hw).expand(n, 1, cv, hw)).squeeze(1)
    else:
        want = vv.double().mean(1)
    got = out.view(n, cv, hw)
    assert rel_err(got[:, :, edge], want[:, :, edge]) <= 1e-6, (kind, path)


# ---------------------------------------------------------------------------------------------------------------------
# 3. bf16 NCHW route
# ---------------------------------------------------------------------------------------------------------------------
def _bf16_problem(n, t, c, cv, h, w, seed):
    q, k, v, _ = _core_problem(n, t, c, cv, h, w, seed)
    return q.bfloat16(), k.bfloat16(), v.bfloat16()


@pytest.mark.parametrize('t', sorted(VEC4_SHAPES))
def test_bf16_kernel_every_reference_count(t):
    """mrapa_attention_bf16 against the fp64 oracle on the same bf16-rounded inputs."""
    n, _, c, cv, h, w = VEC4_SHAPES[t]
    q, k, v = _bf16_problem(n, t, c, cv, h, w, seed=40 + t)
    out, ran = _traced(lambda: FU.mrapa_attention_bf16(q, k, v, t))
    assert _mrapa(ran) == _expect(f'mrapa_fwd_vec4_kernel<{t}, __nv_bfloat16>'), sorted(ran)
    assert out.dtype == torch.bfloat16 and tuple(out.shape) == (n, cv, h, w)
    ref = oracle.mrapa_attention_oracle(q, k, v, t, dtype=torch.float64)
    assert rel_err(out, ref) <= BF16_TOL, rel_err(out, ref)


@pytest.mark.parametrize('c', [64, 128, 256])
def test_bf16_channels_last_training_path_vs_fp64(c):
    """The autograd Function on bf16 channels-last tensors (the convolutions' outputs under autocast) at t = 5: values
    and gradients against fp64 autograd through the oracle on the same bf16 inputs."""
    n, t, h, w = 2, 5, 12, 20
    cl = torch.channels_last
    q, k, v = _bf16_problem(n, t, c, 2 * c, h, w, seed=50 + c)
    go = _randn(torch.Generator(device=DEV).manual_seed(c), n, 2 * c, h, w).bfloat16()
    leaves = [x.contiguous(memory_format=cl).requires_grad_(True) for x in (q, k, v)]

    def run():
        out = M.mrapa_attention(leaves[0], leaves[1], leaves[2], t)
        return out.detach(), torch.autograd.grad(out, leaves, go.contiguous(memory_format=cl))
    (out, grads), ran = _traced(run)
    assert _mrapa(ran) == _expect('mrapa_fwd_vec4_kernel<5, float>', 'mrapa_bwd_vec4_kernel<5>'), sorted(ran)
    assert out.dtype == torch.bfloat16 and out.is_contiguous(memory_format=cl)
    ref, rgrads = _oracle_fwd_bwd(q, k, v, go, t)
    assert rel_err(out, ref) <= BF16_TRAIN_TOL, rel_err(out, ref)
    for x, r, name in zip(grads, rgrads, ('emb_t', 'emb', 'ass')):
        assert x.dtype == torch.bfloat16 and x.is_contiguous(memory_format=cl), name
        assert rel_err(x, r) <= BF16_TRAIN_TOL, (name, rel_err(x, r))


BF16_ROUTES = {   # name: (n, t, C, Cv, h, w), misaligned input, kernel the public entry has to take
    'aligned_t5': ((2, 5, 32, 64, 8, 12), False, 'mrapa_fwd_vec4_kernel<5, __nv_bfloat16>'),
    't9': ((2, 9, 32, 64, 8, 12), False, 'mrapa_fwd_kernel<16>'),
    't12': ((1, 12, 16, 32, 10, 10), False, 'mrapa_fwd_kernel<16>'),
    't16': ((2, 16, 24, 48, 6, 10), False, 'mrapa_fwd_kernel<16>'),
    'grid7x9': ((2, 5, 64, 128, 7, 9), False, 'mrapa_fwd_kernel<8>'),
    'misaligned': ((2, 5, 32, 64, 8, 12), True, 'mrapa_fwd_vec4_kernel<5, float>'),
}


@pytest.mark.parametrize('case', list(BF16_ROUTES))
def test_bf16_inference_route(case):
    """Three bf16 tensors without autograd: the public entry takes the bf16-I/O kernel where it serves the call and the
    fp32 kernels otherwise (more than 8 references, h*w % 4 != 0, a plane that is not 8-byte aligned), returning bf16
    within the bf16 bound either way.  mrapa_attention_bf16 itself refuses those calls."""
    (n, t, c, cv, h, w), mis, kernel = BF16_ROUTES[case]
    q, k, v = _bf16_problem(n, t, c, cv, h, w, seed=60)
    if mis:
        k = _misaligned(k)
    with torch.no_grad():
        out, ran = _traced(lambda: M.mrapa_attention(q, k, v, t))
    assert _mrapa(ran) == _expect(kernel), sorted(ran)
    assert out.dtype == torch.bfloat16 and tuple(out.shape) == (n, cv, h, w)
    ref = oracle.mrapa_attention_oracle(q, k, v, t, dtype=torch.float64)
    assert rel_err(out, ref) <= BF16_TOL, rel_err(out, ref)
    if 'bfloat16' not in kernel:
        with pytest.raises(RuntimeError, match='mrapa_attention_forward_bf16'):
            FU.mrapa_attention_bf16(q, k, v, t)


def test_fusion_module_autocast_bf16_nine_references():
    """MRAPAFusion under bf16 autocast without autograd, with 9 references (more than the bf16 kernel serves): runs, and
    agrees with the fp32 module within the bf16 rounding of its six convolutions."""
    torch.manual_seed(0)
    m = M.MRAPAFusion(nf=16, ref_nf=32).to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(1)
    target = _randn(g, 1, 16, 12, 12)
    refs = [_randn(g, 1, 32, 12, 12) for _ in range(9)]
    with torch.no_grad():
        want = m(target, refs)
        with torch.autocast('cuda', torch.bfloat16):
            got = m(target, refs)
    assert got.shape == want.shape and torch.isfinite(got).all()
    assert rel_err(got, want) <= 5e-2, rel_err(got, want)


# ---------------------------------------------------------------------------------------------------------------------
# 4. channels-last inference kernel (bias, PReLU and scale folded in)
# ---------------------------------------------------------------------------------------------------------------------
NHWC_KERNEL = {64: 'mrapa_fwd_nhwc_kernel<2, 1>', 128: 'mrapa_fwd_nhwc_kernel<4, 1>', 256: 'mrapa_fwd_nhwc_kernel<4, 2>'}
# (bias_q, bias_k, bias_v, PReLU weights of q, of k): None = no PReLU, 1 = nn.PReLU() (what MRAPAFusion has), 'C' = one
# weight per channel
NHWC_EPILOGUES = [(True, True, True, 1, 1), (True, True, True, 'C', 'C'), (True, False, False, 'C', 1),
                  (False, True, False, 1, 'C'), (False, False, True, None, None), (False, False, False, None, None)]


def _nhwc_problem(n, t, c, h, w, epi, seed):
    """Raw convolution outputs (channels-last) and the folded epilogue's parameters."""
    g = torch.Generator(device=DEV).manual_seed(seed)

    def cl(*shape):      # [b, C, h, w] channels-last, drawn in NHWC order
        b, ch, hh, ww = shape
        return _randn(g, b, hh, ww, ch).permute(0, 3, 1, 2)
    bq, bk, bv, nq, nk = epi
    q_raw, k_raw, v_raw = cl(n, c, h, w), cl(n * t, c, h, w), cl(n * t, 2 * c, h, w)
    par = dict(bias_q=_randn(g, c, scale=0.5) if bq else None, bias_k=_randn(g, c, scale=0.5) if bk else None,
               bias_v=_randn(g, 2 * c) if bv else None,
               slope_q=None if nq is None else torch.rand(1 if nq == 1 else c, generator=g, device=DEV) * 0.5,
               slope_k=None if nk is None else torch.rand(1 if nk == 1 else c, generator=g, device=DEV) * 0.5,
               q_scale=c ** -0.5)
    return q_raw, k_raw, v_raw, par


def _finished(q_raw, k_raw, v_raw, par, dtype):
    """The epilogues as torch expressions: q = prelu(q_raw + bias_q) * scale, k = prelu(k_raw + bias_k),
    v = v_raw + bias_v, dense NCHW in `dtype`."""
    def fin(x, b, s):
        x = x.to(dtype)
        if b is not None:
            x = x + b.to(dtype).view(1, -1, 1, 1)
        if s is not None:
            x = F.prelu(x, s.to(dtype))
        return x.contiguous()
    return (fin(q_raw, par['bias_q'], par['slope_q']) * par['q_scale'], fin(k_raw, par['bias_k'], par['slope_k']),
            fin(v_raw, par['bias_v'], None))


def _nhwc_grid_warps(total):
    """Pixel-warps of one round of mrapa_fwd_nhwc_kernel's grid-stride loop (mrefsr_mrapa_attention_nhwc's grid: 8 warps
    per CTA, at most 148 * 8 * 4 CTAs)."""
    return min((total + 7) // 8, 148 * 8 * 4) * 8


def _check_nhwc(n, t, c, h, w, epi, seed, min_rounds=1):
    q_raw, k_raw, v_raw, par = _nhwc_problem(n, t, c, h, w, epi, seed)
    out, ran = _traced(lambda: FU.mrapa_attention_nhwc(q_raw, k_raw, v_raw, t, **par))
    assert _mrapa(ran) == _expect(NHWC_KERNEL[c]), sorted(ran)
    assert out.is_contiguous(memory_format=torch.channels_last) and tuple(out.shape) == (n, 2 * c, h, w)
    hw, total = h * w, n * h * w
    nw = _nhwc_grid_warps(total)
    rounds = -(-total // nw)
    assert rounds >= min_rounds, (rounds, min_rounds)
    # fp64 on a pixel subset: first and last pixel of every round and of every image, and a random sample
    px = {0, total - 1}
    for r in range(1, rounds):
        px |= {r * nw - 1, r * nw}
    for i in range(1, n):
        px |= {i * hw - 1, i * hw}
    px |= set(torch.randint(total, (64,), generator=torch.Generator().manual_seed(seed)).tolist())
    px = torch.tensor(sorted(px), device=DEV)
    img, p = px // hw, px % hw
    L = px.numel()
    qs = q_raw.permute(0, 2, 3, 1).reshape(n, hw, c)[img, p].reshape(L, c, 1, 1)
    ks = k_raw.permute(0, 2, 3, 1).reshape(n, t, hw, c)[img, :, p].reshape(L * t, c, 1, 1)
    vs = v_raw.permute(0, 2, 3, 1).reshape(n, t, hw, 2 * c)[img, :, p].reshape(L * t, 2 * c, 1, 1)
    ref = oracle.mrapa_attention_oracle(*_finished(qs, ks, vs, par, torch.float64), t, dtype=torch.float64)
    got = out.permute(0, 2, 3, 1).reshape(total, 2 * c)[px]
    assert rel_err(got, ref.view(L, 2 * c)) <= OUT_TOL, rel_err(got, ref.view(L, 2 * c))
    # every pixel against the fp32 NCHW kernel fed the finished tensors
    want = M.mrapa_attention(*_finished(q_raw, k_raw, v_raw, par, torch.float32), t)
    assert rel_err(out, want) <= OUT_TOL, rel_err(out, want)


@pytest.mark.parametrize('t', range(1, 9))
@pytest.mark.parametrize('c', [64, 128, 256])
def test_nhwc_every_instantiation_and_epilogue(c, t):
    """All three <V, J> instantiations at t = 1..8; the epilogue combination cycles with t, so each channel count meets
    every combination of biases and PReLU weight counts."""
    _check_nhwc(2, t, c, 12, 20, NHWC_EPILOGUES[(t - 1) % len(NHWC_EPILOGUES)], seed=c + t)


@pytest.mark.parametrize('n,t,c,h,w', [(16, 5, 64, 160, 160), (2, 4, 128, 136, 160), (3, 3, 256, 96, 144)])
def test_nhwc_grid_stride_rounds(n, t, c, h, w):
    """More pixels than one round of the capped grid (37 888 pixel-warps): config 2's 16 x 160^2 (11 rounds), and image
    boundaries that fall inside a round."""
    _check_nhwc(n, t, c, h, w, NHWC_EPILOGUES[1], seed=7, min_rounds=2)


def test_nhwc_refusals():
    def call(c, cv, t, nq=1):
        q = torch.zeros(1, c, 4, 4, device=DEV).contiguous(memory_format=torch.channels_last)
        k = torch.zeros(t, c, 4, 4, device=DEV).contiguous(memory_format=torch.channels_last)
        v = torch.zeros(t, cv, 4, 4, device=DEV).contiguous(memory_format=torch.channels_last)
        FU.mrapa_attention_nhwc(q, k, v, t, slope_q=torch.full((nq,), 0.25, device=DEV))
    call(64, 128, 2)
    call(64, 128, 2, nq=64)
    for args in ((96, 192, 2), (64, 64, 2), (64, 256, 2), (64, 128, 9), (64, 128, 2, 2), (64, 128, 2, 63)):
        with pytest.raises(RuntimeError, match='mrefsr_mrapa_attention_nhwc'):
            call(*args)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------
# 5. fusion head under autograd against a float64 copy of the module
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def no_tf32_matmul():
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = old


@pytest.mark.parametrize('layout', ['nchw', 'channels_last'])
@pytest.mark.parametrize('c', [64, 128, 256])
def test_fusion_head_training_vs_fp64(c, layout, no_tf32_matmul, monkeypatch):
    """MRAPAFusion(nf=64, ref_nf=c) at t = 5 in fp32 under autograd (the training step's fusion head; in channels-last
    its convolutions' epilogues run as BiasActFunction) against a CPU float64 copy whose attention core is the oracle:
    output, input gradients and every parameter gradient."""
    n, t, h, w = 2, 5, 12, 16
    torch.manual_seed(c)
    m = M.MRAPAFusion(nf=64, ref_nf=c)
    ref_m = copy.deepcopy(m).double()
    g = torch.Generator().manual_seed(c + 1)
    target, refs = torch.randn(n, 64, h, w, generator=g), torch.randn(n * t, c, h, w, generator=g)
    go = torch.randn(n, 64, h, w, generator=g)
    mf = torch.channels_last if layout == 'channels_last' else torch.contiguous_format
    m = m.to(DEV).to(memory_format=mf)
    xs = [x.to(DEV).contiguous(memory_format=mf).requires_grad_(True) for x in (target, refs)]
    names, params = zip(*m.named_parameters())

    def run():
        y = m.forward_stacked(xs[0], xs[1], t)
        return y.detach(), torch.autograd.grad(y, xs + list(params), go.to(DEV).contiguous(memory_format=mf))
    # no TF32 anywhere; in NCHW torch's own GEMM convolutions instead of cuDNN, whose NCHW algorithms put
    # spatial_attn.weight's gradient 5e-4 and 8e-4 from fp64 at c = 256 / 128 (its channels-last ones stay within 1e-4)
    with torch.backends.cudnn.flags(enabled=layout == 'channels_last', allow_tf32=False):
        (y, grads), ran = _traced(run)
    assert _mrapa(ran) == _expect('mrapa_fwd_vec4_kernel<5, float>', 'mrapa_bwd_vec4_kernel<5>'), sorted(ran)
    epilogue = {'bias_act_train_fwd_kernel<float>', 'bias_act_train_bwd_kernel<float>', 'bias_grad_sum_kernel'}
    if layout == 'channels_last':
        assert epilogue <= ran, sorted(ran)
    else:
        assert not (epilogue & ran), sorted(ran)

    rs = [x.double().requires_grad_(True) for x in (target, refs)]
    with monkeypatch.context() as mp:
        mp.setattr(FU, 'mrapa_attention', lambda q, k, v, tt: oracle.mrapa_attention_oracle(q, k, v, tt))
        y_ref = ref_m.forward_stacked(rs[0], rs[1], t)
    y_ref.backward(go.double())

    got = dict(zip(('target', 'refs') + names, grads))
    want = {'target': rs[0].grad, 'refs': rs[1].grad, **{k: p.grad for k, p in ref_m.named_parameters()}}
    assert got.keys() == want.keys() and all(v is not None for v in want.values())
    y_ref = y_ref.detach()
    assert float((y.cpu().double() - y_ref).norm()) <= 1e-4 * float(y_ref.norm())
    gmax = max(float(v.norm()) for v in want.values())
    for k in want:
        a, b = got[k].cpu().double(), want[k]
        assert float((a - b).norm()) <= 1e-4 * float(b.norm()) + 1e-6 * gmax, (k, float((a - b).norm() / b.norm()))


# ---------------------------------------------------------------------------------------------------------------------
# 6. BiasActFunction at training row counts
# ---------------------------------------------------------------------------------------------------------------------
BIAS_ACT_CASES = {'leaky': (T.ACT_LEAKY, 0.1, False), 'relu': (T.ACT_LEAKY, 0.0, False),
                  'residual': (T.ACT_NONE, 0.0, True), 'bias_only': (T.ACT_NONE, 0.0, False)}


@pytest.mark.parametrize('case', list(BIAS_ACT_CASES))
@pytest.mark.parametrize('shape,dtype', [((12, 64, 160, 160), torch.float32), ((12, 64, 160, 160), torch.bfloat16),
                                         ((60, 256, 40, 40), torch.bfloat16)])
def test_bias_act_training_rows(shape, dtype, case):
    """The training epilogue on a whole training tensor (rows = B*H*W up to 307 200): the backward's grid-stride loop
    takes many rounds and bias_grad_sum_kernel adds more partial rows than it has lanes.  y and grad_in against the
    torch expression; grad_bias against a float64 sum, per channel within 1e-5 * sum|g| (about 95 sequential fp32
    additions per channel); two backward calls give the same grad_bias bit for bit."""
    act, slope, use_res = BIAS_ACT_CASES[case]
    bf16 = dtype == torch.bfloat16
    b, c, h, w = shape
    rows = b * h * w
    rpb = 256 // (c // (8 if bf16 else 4))      # rows per CTA and round of bias_act_train_bwd_kernel
    blocks = M._lib.lib().mrefsr_bias_act_train_blocks()
    assert blocks > 32 and rows > blocks * rpb, (blocks, rows, rpb)
    g = torch.Generator(device=DEV).manual_seed(5)

    def cl():
        return _randn(g, b, h, w, c).permute(0, 3, 1, 2).to(dtype)
    x0, r0, go = cl(), cl(), cl()
    b0 = _randn(g, c)
    x, r, bias = x0.clone().requires_grad_(True), r0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    inputs = [x, bias] + ([r] if use_res else [])

    def run():
        y = T.BiasActFunction.apply(x * 1.0, bias, act, slope, r if use_res else None, 1.0)
        grads = torch.autograd.grad(y, inputs, go, retain_graph=True)
        gb2, = torch.autograd.grad(y, bias, go)
        return y.detach(), grads, gb2
    (y, grads, gb2), ran = _traced(run)
    tn = '__nv_bfloat16' if bf16 else 'float'
    assert {f'bias_act_train_fwd_kernel<{tn}>', f'bias_act_train_bwd_kernel<{tn}>', 'bias_grad_sum_kernel'} <= ran
    gx, gb = grads[0], grads[1]
    assert torch.equal(gb, gb2)
    if use_res:
        assert torch.equal(grads[2], go)

    # y and grad_in: the torch expression the Function replaces (bounds of test_trunk_gpu's small-shape test)
    tol = 1.6e-2 if bf16 else 1e-6
    xr, rr = x0.clone().requires_grad_(True), r0.clone().requires_grad_(True)
    yr = xr.float() + b0.view(1, -1, 1, 1)
    if bf16:
        yr = yr.to(dtype).float()
    if act == T.ACT_LEAKY:
        yr = F.leaky_relu(yr, slope)
    if use_res:
        yr = yr + rr.float()
    yr = yr.to(dtype)
    gxr, = torch.autograd.grad(yr, xr, go)
    assert rel_err(y, yr) <= tol, rel_err(y, yr)
    assert rel_err(gx, gxr) <= tol, rel_err(gx, gxr)

    # grad_bias: fp64 sum over the rows of the gradient after the activation (its mask from the stored output)
    ge = go.double()
    if act == T.ACT_LEAKY:
        ge = torch.where(y > 0, ge, ge * slope)
    want = ge.sum((0, 2, 3))
    bound = 1e-5 * ge.abs().sum((0, 2, 3))
    err = (gb.double() - want).abs()
    assert (err <= bound).all(), float((err / bound).max())
