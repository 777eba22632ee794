#!/usr/bin/env python
"""bench.py -- throughput of MRefSR's reference-alignment hot path on B200 (this repo) or on host cores
(--impl reference: the CPU oracle port of the reference algorithm).

One "step" = one pass of the hot path over one batch of synthetic CUFED5-shaped input, BASELINE.json config 2:
B images per GPU (default 16), R = 5 references, 160x160 HR (feature grids 40/80/160, C = 256/128/64):
  (1) correspondence matcher over the B*R (image, reference) pairs (+ per-pixel normalisation, + pre-offsets
      at three scales),
  (2) DynAgg offset/mask assembly + DCNv2 forward at three scales over the B*R samples,
  (3) multi-reference attention fusion at three scales.
metric = x4 SR images/sec through that path (images = B per step).  Multi-GPU: images are independent, so the
batch is sharded across ranks with no data-path collective ("weak" scaling: B per GPU fixed).

Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement" for the definitions of every key.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'x4 SR images/sec through the reference-alignment hot path (match + DCNv2 + fusion), 5 refs @160^2 HR'
UNIT = 'images/s'
SCALES = ((256, 40), (128, 80), (64, 160))   # (channels, feature grid) at relu3_1 / relu2_1 / relu1_1
DG = 8


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=16, help='images per GPU per step')
    ap.add_argument('--refs', type=int, default=5)
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-images', type=int, default=2, help='images in the bounded CPU-baseline sample')
    ap.add_argument('--match-mode', default='auto')
    ap.add_argument('--dcn-mode', default='auto')
    ap.add_argument('--no-full-model', action='store_true', help='skip the whole-network (images in -> SR out) leg')
    ap.add_argument('--no-extras', action='store_true',
                    help='skip the extra legs (sustained run, GPU reference route, configs 3 / 4 / 5)')
    ap.add_argument('--no-fused', action='store_true',
                    help='materialise pre-offsets / offset / mask (reference operator boundaries) instead of the '
                         'fused DynAgg gather')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the outputs of the last one as DIR/<name>.npy (rank 0; below 64 MB '
                         'in all: a larger output is sampled at fixed seeded positions)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    return args


# ----------------------------------------------------------------------------------------------------------
# synthetic workload
# ----------------------------------------------------------------------------------------------------------
def make_inputs(b, r, seed, device, pin=False):
    """Seeded synthetic tensors of the config-2 shapes.  Returned on `device` ('cpu' tensors are pinned if pin)."""
    g = torch.Generator().manual_seed(seed)

    def rnd(*shape, scale=1.0):
        t = torch.randn(*shape, generator=g) * scale
        if device != 'cpu':
            return t.to(device)
        return t.pin_memory() if pin else t

    # matcher features (SURVEY.md section 8d): each image gets references that are integer translations of itself
    # (known arg-max, similarity ~ 1), independent references (near-tie stress) and one zero-padded reference
    # (exact-tie plateau, like CUFED5's pad-to-500^2)
    big = torch.randn(b, 256, 48, 48, generator=g)
    fin = big[:, :, 4:44, 4:44].contiguous()
    refs = []
    for k in range(r):
        kind = k % 5
        if kind == 0:
            ref = big[:, :, 3:43, 2:42]
        elif kind == 1:
            ref = big[:, :, 7:47, 5:45]
        elif kind == 4:
            ref = big[:, :, 2:42, 6:46].clone()
            ref[:, :, 30:, :] = 0
            ref[:, :, :, 32:] = 0
        else:
            ref = torch.randn(b, 256, 40, 40, generator=g)
        refs.append(ref)
    fref = torch.stack(refs, 1).reshape(b * r, 256, 40, 40).contiguous()

    def place(t):
        if device != 'cpu':
            return t.to(device)
        return t.pin_memory() if pin else t

    d = {'feat_in': place(fin), 'feat_ref': place(fref)}
    for c, hw in SCALES:
        d[f'x{c}'] = rnd(b * r, c, hw, hw)                          # reference VGG features (DCN input)
        d[f'conv_out{c}'] = rnd(b * r, 3 * DG * 9, hw, hw, scale=0.5)  # raw conv_offset_mask output
        d[f'w{c}'] = rnd(c, c, 3, 3, scale=(c * 9) ** -0.5)
        d[f'b{c}'] = rnd(c, scale=0.1)
        d[f'emb_t{c}'] = rnd(b, c, hw, hw, scale=0.2)
        d[f'emb{c}'] = rnd(b * r, c, hw, hw)
        d[f'ass{c}'] = rnd(b * r, 2 * c, hw, hw)
    return d


def input_bytes(d):
    return sum(t.numel() * t.element_size() for t in d.values())


def hot_path_step(M, d, b, r, match_mode, dcn_mode, fused=True):
    """One pass over the batch on the current stream.  Returns the list of outputs."""
    from mrefsr_b200.dynagg import DynAggOffsetsFunction
    from mrefsr_b200.dcn import dcn_forward_raw, dynagg_dcn_forward
    outs = []
    idx, val = M.feature_match_index_batched(d['feat_in'], d['feat_ref'], is_norm=True, norm_input=True,
                                             normalize_pixels=True, in_div=r, mode=match_mode)
    outs += [idx, val]
    pre = None if fused else M.pre_offsets(idx)                # [B*R,9,s*40,s*40,2] for s = 1, 2, 4
    for k, (c, hw) in enumerate(SCALES):
        if fused:   # offsets / masks / pre-offsets assembled inside the DCN gather
            y = dynagg_dcn_forward(d[f'x{c}'], d[f'conv_out{c}'], idx, hw // 40, d[f'w{c}'], d[f'b{c}'], DG)
        else:       # the reference's operator boundaries, one kernel each
            off, mask = DynAggOffsetsFunction.apply(d[f'conv_out{c}'], pre[k], DG, None)
            y = dcn_forward_raw(d[f'x{c}'], off, mask, d[f'w{c}'], d[f'b{c}'], (1, 1), (1, 1), (1, 1), 1, DG,
                                mode=dcn_mode)
        f = M.mrapa_attention(d[f'emb_t{c}'], d[f'emb{c}'], d[f'ass{c}'], r)
        outs += [y, f]
    return outs


OUTPUT_NAMES = ('match_index', 'match_similarity', 'dcn_relu3_1', 'fusion_relu3_1', 'dcn_relu2_1', 'fusion_relu2_1',
                'dcn_relu1_1', 'fusion_relu1_1')   # hot_path_step's outputs, in order
DUMP_BYTES = 60 << 20           # all the .npy files together stay below 64 MB


def dump_outputs(outs, out_dir):
    """Write hot_path_step's outputs as out_dir/<name>.npy: floating outputs as float32, integer ones as float64 (exact).
    An output larger than its share of DUMP_BYTES is stored as the values at a sorted sample of flat (logical NCHW)
    positions drawn from a generator seeded by the output's place in the list, so that two runs with the same
    arguments, on any build, store the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // len(outs)
    for k, (name, t) in enumerate(zip(OUTPUT_NAMES, outs, strict=True)):
        dt = torch.float32 if t.is_floating_point() else torch.float64
        n = share // dt.itemsize
        if t.numel() > n:
            pos = torch.randint(t.numel(), (n,), generator=torch.Generator().manual_seed(k)).sort().values
            t = t.flatten()[pos.to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().to(dt).cpu().contiguous().numpy())


# ----------------------------------------------------------------------------------------------------------
# algorithmic work (DESIGN.md "Measurement"; SURVEY.md section 8d)
# ----------------------------------------------------------------------------------------------------------
def algorithmic(b, r):
    n = 38 * 38
    w = {'match_main': {'flops': 2.0 * n * n * 2304 * b * r, 'bytes': (2 * 256 * 1600 * 4 + 12 * n) * b * r}}
    dcn_f = sum(2.0 * c * c * 9 * hw * hw for c, hw in SCALES) * b * r
    dcn_b = sum(4.0 * hw * hw * (c + 27 * DG + c) + 4.0 * c * c * 9 + 4 * c for c, hw in SCALES) * b * r
    w['dcn_fwd'] = {'flops': dcn_f, 'bytes': dcn_b}
    w['fusion_fwd'] = {'flops': 0.0, 'bytes': sum(4.0 * hw * hw * c * (3 + 3 * r) for c, hw in SCALES) * b}
    return w


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        j = json.load(open(p))
        return {'hbm_gbs': j['hbm_gbs'], 'bf16_tflops': j['bf16_tflops'],
                'bf16_tflops_sustained': j.get('bf16_tflops_sustained', j['bf16_tflops']), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        sm.sort()
        # median of the samples in the upper half = clocks under load (idle samples before/after drag it down)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {'sm_mhz': med, 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


# ----------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference algorithm, all host threads
# ----------------------------------------------------------------------------------------------------------
def cpu_hot_path(n_images, r, seed=4321):
    """One pass of the same hot path for n_images images on the host (oracle port; see oracle/__init__.py)."""
    import torch.nn.functional as F
    import oracle
    from oracle.dcn import modulated_deform_conv_c
    d = make_inputs(n_images, r, seed, 'cpu')
    t0 = time.perf_counter()
    idxs = []
    for p in range(n_images * r):
        a = F.normalize(d['feat_in'][p // r].reshape(256, -1), dim=0).view(256, 40, 40)
        q = F.normalize(d['feat_ref'][p].reshape(256, -1), dim=0).view(256, 40, 40)
        idx, _ = oracle.feature_match_index_oracle(a, q, is_norm=True, norm_input=True, use_conv=True)
        idxs.append(idx)
    t1 = time.perf_counter()
    pres = [oracle.pre_offsets_oracle(i) for i in idxs]
    t_dcn = t_fus = 0.0
    for (c, hw), key in zip(SCALES, ('relu3_1', 'relu2_1', 'relu1_1')):
        ta = time.perf_counter()
        pre = torch.stack([p[key] for p in pres], 0)
        off, mask = oracle.dynagg_offsets_oracle(d[f'conv_out{c}'], pre, DG)
        modulated_deform_conv_c(d[f'x{c}'], off, mask, d[f'w{c}'], d[f'b{c}'], 1, 1, 1, 1, DG)
        tb = time.perf_counter()
        oracle.mrapa_attention_oracle(d[f'emb_t{c}'], d[f'emb{c}'], d[f'ass{c}'], r)
        tc = time.perf_counter()
        t_dcn += tb - ta
        t_fus += tc - tb
    t2 = time.perf_counter()
    return {'total_s': t2 - t0, 'match_s': t1 - t0, 'dcn_s': t_dcn, 'fusion_s': t_fus}


def _set_omp_threads(n):
    import ctypes
    for name in ('libgomp.so.1', 'libomp.so', 'libiomp5.so'):
        try:
            ctypes.CDLL(name).omp_set_num_threads(int(n))
        except OSError:
            pass


def cpu_baseline(n_images, r):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    _set_omp_threads(cores)                             # torchrun exports OMP_NUM_THREADS=1; the C DCN port uses OpenMP
    cpu_hot_path(1, r)                                  # warm-up (thread pools, page faults)
    best = min((cpu_hot_path(n_images, r) for _ in range(2)), key=lambda x: x['total_s'])
    return {'value': n_images / best['total_s'], 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': '%d image(s) x %d refs @160^2 through the oracle port (torch CPU matcher + OpenMP C DCN + '
                      'torch CPU fusion), best of 2' % (n_images, r),
            'split_s': {k: round(v, 4) for k, v in best.items()}}


def run_reference(args):
    """--impl reference: the reference algorithm's CPU implementation (oracle port; /root/reference is a Python
    tree that cannot travel to the GPU box) on all host cores; each step = a bounded sample of the workload."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    _set_omp_threads(cores)
    n_img = 2
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_hot_path(n_img, args.refs)
    steps = args.steps
    # the timed region is the hot path itself (cpu_hot_path's own clock), as in the GPU arm, whose inputs also
    # exist before the clock starts: drawing the synthetic tensors (0.4 GB of randn per image) is not part of it
    dt = sum(cpu_hot_path(n_img, args.refs)['total_s'] for _ in range(steps))
    v = n_img * steps / dt
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
            'warmup': 1, 'ms_per_step': dt / steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'MRefSR x4 alignment hot path, %d refs @160^2 HR (BASELINE config 2 shapes), '
                                   'bounded sample: %d images per step on host cores' % (args.refs, n_img)},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                             'sample': '%d images x %d refs per step through the oracle port (torch CPU matcher + OpenMP C DCN + torch CPU fusion), %d steps' % (n_img, args.refs, steps)},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def full_model_leg(dev, b, r, rank, world, dist, barrier, steps=5):
    from mrefsr_b200.models import MRefSRPipeline
    torch.manual_seed(10)
    net = MRefSRPipeline().eval().to(dev).channels_last_()     # cuDNN's native layout for the plain convolutions
    torch.backends.cudnn.benchmark = True
    g = torch.Generator().manual_seed(99 + rank)
    lq = torch.rand(b, 3, 40, 40, generator=g).pin_memory()
    up = torch.nn.functional.interpolate(lq, scale_factor=4, mode='bicubic', align_corners=False).clamp(0, 1).pin_memory()
    refs = torch.rand(b, r, 3, 160, 160, generator=g).pin_memory()

    sr_host = torch.empty(b, 3, 160, 160).pin_memory()
    try:
        runner = net.graphed(lq, up, refs)      # CUDA-graph replay: the host launches one graph per batch
        graphed = True

        def step():                              # pinned host images in -> pinned host SR out, every step
            return runner(lq, up, refs, out=sr_host)
    except Exception:  # noqa: BLE001  (a failed capture must not desynchronise the ranks: same steps, launched eagerly)
        torch.cuda.synchronize()
        graphed = False

        def step():
            sr = net(lq.to(dev, non_blocking=True), up.to(dev, non_blocking=True), refs.to(dev, non_blocking=True))
            return sr_host.copy_(sr, non_blocking=True)
    for _ in range(4):
        step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        out = step()
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    h2d = sum(t.numel() * 4 for t in (lq, up, refs))
    return {'value': b * world * steps / float(dt.item()), 'unit': UNIT, 'ms_per_step': float(dt.item()) / steps * 1e3,
            'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': out.numel() * 4, 'steps': steps,
            'note': 'whole x4 MRefSR network, random-init weights, host images in -> SR images out; '
                    'convolutions = cuDNN (TF32 allowed, channels_last), bias / activation / residual epilogues, '
                    'layout hand-offs and the alignment path = this library; ' +
                    ('the forward is replayed as one CUDA graph' if graphed else 'launched eagerly (graph capture failed)')}


# ----------------------------------------------------------------------------------------------------------
def _guard_stdout():
    """stdout carries exactly one JSON line.  Libraries write there too (NCCL_DEBUG=INFO prints its log on stdout), so
    file descriptor 1 is pointed at stderr for the whole run and the line is written to the saved descriptor."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, 'w')


def gpu_reference_leg(b, r):
    """SURVEY 8(d) GPU-side comparison set: the reference's own GPU route (per-pair unfold + cuDNN conv2d matcher, DynAgg
    glue in torch, DCN through the reference's deform_conv_ext compiled unmodified for sm_100a and through torchvision,
    fusion as written) on the same inputs in the same run.  It lives in tests/ (it loads the checker build oracle/_ref)
    and runs as a subprocess; this function only relays its summary line."""
    script = os.path.join(ROOT, 'tests', 'perf_reference_gpu.py')
    try:
        p = subprocess.run([sys.executable, script, '--batch', str(b), '--refs', str(r)], capture_output=True, text=True,
                           timeout=600, cwd=ROOT)
        lines = [json.loads(ln) for ln in p.stdout.splitlines() if ln.startswith('{')]
        summ = [ln for ln in lines if ln.get('what') == 'summary']
        if p.returncode != 0 or not summ:
            return {'error': (p.stderr or p.stdout)[-300:]}
        out = dict(summ[-1])
        out.pop('what', None)
        out['dcn_per_scale'] = [{k: ln[k] for k in ('C', 'hw', 'dcn_ref_ext_ms', 'dcn_torchvision_ms', 'glue_ref_ms',
                                                    'ours_fused_ms', 'rel_diff_vs_torchvision')}
                                for ln in lines if ln.get('what') == 'dcn']
        out['note'] = ('reference route = what a wdmwhh/MRefSR user runs on this GPU today (stock PyTorch ops; DCN = the '
                       "faster of the reference's own extension built for sm_100a and torchvision); same inputs")
        return out
    except Exception as e:  # noqa: BLE001
        return {'error': repr(e)[:300]}


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    out_stream = _guard_stdout()

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; the product path has no CPU fallback '
                         '(use --impl reference for the CPU baseline)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    dist = None
    if world > 1:
        # NCCL_DEBUG is left alone: whatever NCCL prints goes to stderr (_guard_stdout), stdout stays one JSON line
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group('nccl', device_id=dev)

    import mrefsr_b200 as M
    from mrefsr_b200 import _lib
    b, r = args.batch, args.refs
    fused = not args.no_fused
    d = make_inputs(b, r, 1234 + rank, dev)
    in_gb = input_bytes(d) / 1e9

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up
    for _ in range(max(3, args.warmup)):
        hot_path_step(M, d, b, r, args.match_mode, args.dcn_mode, fused)
    barrier()

    # ---- timed region: K steps, device-timed, inputs resident in HBM (several GB/step of inputs >> 126 MB L2)
    _lib.timing_enable(True)
    _lib.timing_read()
    launches0 = _lib.launch_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps - 1):
        hot_path_step(M, d, b, r, args.match_mode, args.dcn_mode, fused)
    outs = hot_path_step(M, d, b, r, args.match_mode, args.dcn_mode, fused)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    launches = _lib.launch_count() - launches0
    ktimes = _lib.timing_read()
    _lib.timing_enable(False)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = b * world * args.steps / (ms_max / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(outs, args.dump_outputs)
    del outs

    # ---- sustained: the same step back to back for >= 3 s (the timed region above is a fraction of a second)
    extras = {}
    if not args.no_extras:
        sys.path.insert(0, os.path.join(ROOT, 'tools'))
        import bench_legs
        try:
            extras['sustained'] = bench_legs.sustained_leg(
                lambda: hot_path_step(M, d, b, r, args.match_mode, args.dcn_mode, fused), b,
                ClockSampler if rank == 0 else None, local_rank, dev, dist)
        except Exception as e:  # noqa: BLE001
            extras['sustained'] = {'error': repr(e)[:200]}

    # ---- e2e: same step through the operator API with HOST (pinned) buffers, H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        # allocation may fail on a crowded host (pinned memory: 6.3 GB per rank) -- decide collectively, so that no
        # rank is left waiting in a barrier
        alloc_err = None
        try:
            hd = make_inputs(b, r, 1234 + rank, 'cpu', pin=True)
            h2d = input_bytes(hd)
            del d
            torch.cuda.empty_cache()
            dev_in = [{k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in hd.items()} for _ in range(2)]
        except Exception as e:  # noqa: BLE001
            alloc_err = repr(e)[:200]
        ok = torch.tensor([0 if alloc_err else 1], dtype=torch.int32, device=dev)
        if dist is not None:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if not args.no_e2e and int(ok.item()) == 0:
        e2e = {'error': alloc_err or 'allocation failed on another rank'}
    elif not args.no_e2e:
        d2h = [0]
        copy_in, copy_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        cur = torch.cuda.current_stream(dev)
        # Double-buffered pipeline over steps: while step i computes and its results stream back to the host
        # (PCIe is full duplex), the inputs of step i+1 are already crossing the bus into the second buffer set.
        # Every step still pays its own H2D of all inputs and its own D2H of all results inside the timed region.
        host_out = [None, None]
        in_ready = [torch.cuda.Event(), torch.cuda.Event()]
        in_free = [torch.cuda.Event(), torch.cuda.Event()]
        out_done = [torch.cuda.Event(), torch.cuda.Event()]

        def h2d_issue(i):
            s_ = i & 1
            with torch.cuda.stream(copy_in):
                copy_in.wait_event(in_free[s_])          # the step that last read this buffer set has finished
                for k, v in hd.items():
                    dev_in[s_][k].copy_(v, non_blocking=True)
                in_ready[s_].record(copy_in)

        def e2e_run(n):
            for e in in_free:
                e.record(cur)
            h2d_issue(0)
            for i in range(n):
                s_ = i & 1
                if i + 1 < n:
                    h2d_issue(i + 1)
                cur.wait_event(in_ready[s_])
                outs = hot_path_step(M, dev_in[s_], b, r, args.match_mode, args.dcn_mode, fused)
                in_free[s_].record(cur)
                done = torch.cuda.Event()
                done.record(cur)
                with torch.cuda.stream(copy_out):
                    copy_out.wait_event(done)
                    if host_out[s_] is None:
                        host_out[s_] = [torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs]
                    else:
                        out_done[s_].synchronize()       # host buffers of step i-2 have been filled
                    for h_, o in zip(host_out[s_], outs):
                        h_.copy_(o, non_blocking=True)
                        o.record_stream(copy_out)
                    out_done[s_].record(copy_out)
                d2h[0] = sum(o.numel() * o.element_size() for o in outs)
            copy_out.synchronize()
            torch.cuda.synchronize()
        e2e_run(2)
        barrier()
        n_e2e = max(4, min(args.steps, 8))
        t0 = time.perf_counter()
        e2e_run(n_e2e)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {'value': b * world * n_e2e / float(dt.item()), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
               'd2h_bytes_per_step': d2h[0], 'steps': n_e2e,
               'note': 'pinned host tensors -> operator API -> pinned host results, double-buffered over steps '
                       '(H2D of step i+1 overlaps compute + D2H of step i; the first H2D is exposed); '
                       'PCIe-bound at this operator boundary'}

    # ---- full model: the whole x4 MRefSR network (extractor -> matcher -> VGG19 -> MRAPARestorationNet) from pinned
    # host images to SR images on the host; plain convolutions are cuDNN (TF32 allowed, torch default), the alignment
    # path is this repo's kernels.  Extra information next to the contract keys: the literal "x4 SR images/sec".
    full = None
    if not args.no_full_model:
        try:
            full = full_model_leg(dev, b, r, rank, world, dist, barrier)
        except Exception as e:  # noqa: BLE001
            full = {'error': repr(e)[:200]}

    # ---- extra legs: BASELINE configs 3 / 4 / 5 and the reference's GPU route, in the driver's record
    if not args.no_extras:
        torch.cuda.empty_cache()
        for name, fn in (('ragged', lambda: bench_legs.ragged_leg(dev, rank, world, dist)),
                         ('train_step', lambda: bench_legs.train_step_leg(dev, rank, world, dist)),
                         ('refshard', lambda: bench_legs.refshard_leg(dev, rank, world, dist))):
            # an exception on one rank only would leave the others in a collective: legs catch nothing themselves,
            # every rank runs the same code on the same shapes, so a failure is common to all ranks
            try:
                extras[name] = fn()
            except Exception as e:  # noqa: BLE001
                extras[name] = {'error': repr(e)[:300]}
            torch.cuda.empty_cache()
        if world == 1 and rank == 0:
            torch.cuda.synchronize()
            extras['gpu_reference'] = gpu_reference_leg(b, r)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (by measured device time inside the timed region)
    pk = peaks()
    work = algorithmic(b, r)
    per_kernel = {}
    for k, (tot_ms, n) in ktimes.items():
        if n:
            per_kernel[k] = {'ms_per_step': tot_ms / args.steps, 'launches_per_step': n / args.steps}
    dom = max((k for k in per_kernel if k in work), key=lambda k: per_kernel[k]['ms_per_step'])

    traffic = {}
    tp = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(tp) and b == 16 and r == 5 and fused:     # measured for exactly this workload
        traffic = json.load(open(tp)).get('bytes_per_step', {})

    def roof(k):
        t_s = per_kernel[k]['ms_per_step'] / 1e3
        wk = work[k]
        t_flop = wk['flops'] / (pk['bf16_tflops_sustained'] * 1e12)
        t_byte = wk['bytes'] / (pk['hbm_gbs'] * 1e9)
        if t_flop >= t_byte:
            a = wk['flops'] / t_s / 1e12
            return {'kernel': k, 'bound': 'tensor', 'achieved': a, 'peak': pk['bf16_tflops_sustained'], 'unit': 'TFLOP/s',
                    'frac': a / pk['bf16_tflops_sustained'], 'traffic': traffic.get(k),
                    'peak_source': pk['source'] + ' (cuBLAS bf16, sustained)'}
        a = wk['bytes'] / t_s / 1e9
        return {'kernel': k, 'bound': 'hbm', 'achieved': a, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                'frac': a / pk['hbm_gbs'], 'traffic': traffic.get(k), 'algorithmic_bytes': wk['bytes'],
                'peak_source': pk['source'] + ' (copy)'}

    roofline = roof(dom)
    roofline['ms_per_launch'] = per_kernel[dom]['ms_per_step'] / per_kernel[dom]['launches_per_step']
    roof_all = {k: roof(k) for k in per_kernel if k in work}
    if 'match_main' in roof_all and args.match_mode in ('auto', 'bf16x3'):
        # The matcher's `achieved` counts the REFERENCE formulation (2 N^2 9C per pair).  Since round 2 the kernel runs the
        # diagonal form: the tensor core computes only the tap-column sums (K = 3C) and the epilogue adds the three
        # tap-row terms, i.e. a third of those MACs -- so the algorithmic fraction can exceed 1.  What the tensor pipe
        # really executes (3 split-bf16 passes on 128 x 256 accumulator tiles that own 120 x 254 outputs):
        rows = (40 - 3) * 40 + 38
        items = b * r * -(-rows // 120) * -(-rows // 254)
        exe = 3 * 2.0 * 128 * 256 * (3 * 256) * items
        t_s = per_kernel['match_main']['ms_per_step'] / 1e3
        roof_all['match_main'].update({
            'executed_tflops': exe / t_s / 1e12, 'executed_flops': exe,
            'executed_frac_of_measured_peak': exe / t_s / 1e12 / pk['bf16_tflops_sustained'],
            'executed_frac_of_nominal_dense_bf16': exe / t_s / 1e12 / 2250.0,
            'note': 'achieved / frac count the reference formulation (9 taps as MACs); the diagonal-form kernel executes a '
                    'third of them (tap-column sums on the tensor core, tap-row sums by warp shuffle in the epilogue), '
                    'in 3 split-bf16 passes'})

    # The DCN's HBM fraction is low by construction in fp32: every sampling point is four scattered 32-byte
    # sectors, 6.7x the algorithmic bytes through L1.  Its practical ceiling is the bilinear gather alone, measured
    # on B200 by tools/micro/gather_bench.cu (64 warps/SM, no MMA; profiles/r01_dcn_gather_microbench.txt):
    # 0.353 / 0.794 / 2.066 ms per 80 samples at the three scales.  Reported next to the HBM roofline, not instead.
    if 'dcn_fwd' in per_kernel:
        floor_ms = (0.353 + 0.794 + 2.066) * (b * r) / 80.0
        roof_all['dcn_fwd']['l1_gather'] = {
            'bound': 'l1-sector gather (microbenchmark of the gather alone, same shapes)', 'floor_ms': floor_ms,
            'achieved_ms': per_kernel['dcn_fwd']['ms_per_step'], 'frac': floor_ms / per_kernel['dcn_fwd']['ms_per_step'],
            'sectors_per_step': 4.0 * 9 * (b * r) * sum(hw * hw * c / 8 for c, hw in SCALES)}
        # Round 2 (profiles/r02_dcn_window.md): ablating the kernel shows that neither HBM nor the L1 gather bounds it -- a
        # free corner fetch saves 0.75 of 3.63 ms.  What does is instruction issue and hand-off latency: the operator
        # needs ~75 instructions per decoded sampling point (position, deform group, tap) and ~70 per gathered
        # 8-channel item (position, chunk, tap).  That count at 100 % issue rate (4 warp instructions per clock per SM
        # at the measured SM clock) is the floor reported here.
        sm_ghz = ((clocks or {}).get('sm_mhz') or 1900.0) / 1e3
        warp_instr = sum((75.0 * DG + 70.0 * c / 8) * 9 * hw * hw for c, hw in SCALES) * (b * r) / 32.0
        floor_issue_ms = warp_instr / (148 * 4 * sm_ghz * 1e9) * 1e3
        roof_all['dcn_fwd']['issue_floor'] = {
            'bound': 'instruction issue: essential decode + gather instructions at 4 warp-instructions/clk/SM',
            'warp_instructions_per_step': warp_instr, 'floor_ms': floor_issue_ms,
            'achieved_ms': per_kernel['dcn_fwd']['ms_per_step'], 'frac': floor_issue_ms / per_kernel['dcn_fwd']['ms_per_step'],
            'note': 'ablation: pipeline skeleton 0.60 + decode 0.49 + gather 0.58 + epilogue stores 0.25 + MMA 0.14 ms add up '
                    'serially at the large scale (profiles/r02_dcn_window.md)'}
        if dom == 'dcn_fwd':
            roofline['l1_gather'] = roof_all['dcn_fwd']['l1_gather']
            roofline['issue_floor'] = roof_all['dcn_fwd']['issue_floor']

    # contract: the CPU baseline is timed on rank 0 at N = 1 only (at N > 1 the host cores are shared by the ranks)
    cpu = None if (args.no_cpu_baseline or world > 1) else cpu_baseline(args.cpu_images, r)

    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': max(3, args.warmup), 'ms_per_step': ms_max / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 I/O (matcher: split-bf16 x3 operands on tcgen05, fp32 accumulate, diagonal form; dcn: tf32 operands, fp32 '
                     'accumulate; fusion: fp32)',
            'data': 'synthetic',
            'config': {'workload': 'MRefSR x4 inference alignment hot path, batch %d per GPU, %d refs at 160x160 '
                                   '(BASELINE config 2): %d matcher pairs, DynAgg+DCNv2 x3 scales over %d samples, '
                                   'fusion x3 scales' % (b, r, b * r, b * r),
                       'images_per_step': b * world, 'l2': 'inputs (%.1f GB/step/GPU) larger than the 126 MB L2' % in_gb,
                       'parallelism': 'batch-sharded x%d, no collective' % world,
                       'match_mode': args.match_mode, 'dcn_mode': args.dcn_mode,
                       'dynagg': 'fused gather (conv_out + arg-max map)' if fused else 'materialised offset/mask'},
            'roofline': roofline, 'roofline_all': roof_all, 'kernel_ms_per_step': per_kernel,
            'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clocks, 'full_model': full}
    line.update(extras)
    out_stream.write(json.dumps(line) + '\n')
    out_stream.flush()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
