"""One DynAgg node, forward + backward, at the training step's shapes (12 images x 5 references = 60 samples, dg 8):
the materialised node (DynAggDCNFunction fed the pre-offsets of the arg-max map) against the fused one
(DynAggFusedFunction, offsets / masks built inside the DCN gather from conv_out and max_idx), timed with CUDA events,
alternating, `--repeats` times each.  Inputs as in the bf16 channels-last training step: x fp32 channels-last (the VGG
feature, no gradient), conv_out bf16 channels-last, leaky ReLU and hand-off folded into the node.  The pre-offsets are
made once outside the timed region (the training step makes them once per step, in correspondences()).

  python tools/dynagg_node_bench.py [--batch 60] [--iters 20] [--repeats 3]
Prints one JSON line per (scale, variant, repeat) and a summary line."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mrefsr_b200 as M  # noqa: E402
from mrefsr_b200.dynagg import DynAggDCNFunction, DynAggFusedFunction  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument('--batch', type=int, default=60)
ap.add_argument('--iters', type=int, default=20)
ap.add_argument('--repeats', type=int, default=3)
args = ap.parse_args()

dev = torch.device('cuda', 0)
CL = torch.channels_last
try:
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True, timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    smi = 'unknown'
card = {'device': torch.cuda.get_device_name(dev), 'nvidia_smi': smi}


def make(s, c, hw, dg=8):
    g = torch.Generator().manual_seed(s)
    b, hp = args.batch, hw // s - 2
    x = torch.randn(b, c, hw, hw, generator=g).to(dev).contiguous(memory_format=CL)
    co = (torch.randn(b, 3 * dg * 9, hw, hw, generator=g) * 0.5).to(dev).to(torch.bfloat16).contiguous(memory_format=CL)
    mi = torch.randint(0, hp * hp, (b, hp, hp), generator=g).to(dev)
    w = (torch.randn(c, c, 3, 3, generator=g) * (9 * c) ** -0.5).to(dev)
    bias = torch.zeros(c, device=dev)
    go = torch.randn(b, c, hw, hw, generator=g).to(dev).to(torch.bfloat16).contiguous(memory_format=CL)
    pre = M.pre_offsets(mi, scales=(s,))[0]
    return x, co, mi, pre, w, bias, go


def run(fused, t, s, dg=8):
    x, co, mi, pre, w, bias, go = t
    co_ = co.detach().requires_grad_(True)
    w_ = w.detach().requires_grad_(True)
    b_ = bias.detach().requires_grad_(True)
    if fused:
        y = DynAggFusedFunction.apply(x, co_, mi, s, w_, b_, dg, 0.1, True)
    else:
        stats = torch.zeros(1, device=dev)
        y = DynAggDCNFunction.apply(x, co_, pre, w_, b_, dg, stats, 0.1, True)
    y.backward(go)


def timed(fused, t, s):
    for _ in range(2):
        run(fused, t, s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.iters):
        run(fused, t, s)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / args.iters


summary = {}
for s, c, hw in ((1, 256, 40), (2, 128, 80), (4, 64, 160)):
    t = make(s, c, hw)
    for rep in range(args.repeats):
        for fused in (False, True):
            ms = timed(fused, t, s)
            name = 'fused' if fused else 'materialised'
            summary.setdefault((s, name), []).append(ms)
            print(json.dumps({'test': 'dynagg_node_fwd_bwd', 'scale': s, 'C': c, 'hw': hw, 'batch': args.batch,
                              'variant': name, 'repeat': rep, 'ms': round(ms, 4)}), flush=True)
    del t
    torch.cuda.empty_cache()
print(json.dumps({'test': 'dynagg_node_summary', **card,
                  'ms_min': {f'{name}_s{s}': round(min(v), 4) for (s, name), v in summary.items()},
                  'ms_max': {f'{name}_s{s}': round(max(v), 4) for (s, name), v in summary.items()}}), flush=True)
