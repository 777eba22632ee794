"""Device times of the DCN modes 'tf32', 'tf32x3' and 'fp32' on the shapes MRefSR runs.

    python tools/dcn_x3_bench.py [--reps N] [--out FILE]

Forward: bench.py's config-2 inputs at its three scales (80 samples = 16 images x 5 references each), the fused
DynAgg entry point (offsets and masks assembled in the gather; no fp32 variant exists) and the operator entry point
on materialised offsets / masks.  Backward: all five gradients at the three DCN shapes of the stage-3 training step
(B 20 / C 64 / 160^2, B 40 / C 128 / 80^2, B 60 / C 256 / 40^2, 8 deform groups), which is what one training step runs.

Every call is timed with CUDA events over a window of `reps` calls after two warm-up calls; the modes alternate,
window by window, three windows each, and the median window is reported (milliseconds per call).  The inputs of every
shape are larger than the 126 MB L2.  Prints one JSON line per (pass, shape, entry point, mode) and a header line with
the GPU's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import mrefsr_b200 as M  # noqa: E402
from mrefsr_b200 import dcn as D  # noqa: E402

DEV = 'cuda:0'
MODES = ('tf32', 'tf32x3', 'fp32')
TRAIN_SHAPES = ((20, 64, 160), (40, 128, 80), (60, 256, 40))


def _gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        q = 'n/a'
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q)


def _window(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / reps


def _time_modes(calls, reps, windows=3):
    """calls: {mode: fn}.  Median over `windows` alternating windows of ms per call."""
    for mode, fn in calls.items():
        with _mode(mode):
            fn()
            fn()
    torch.cuda.synchronize()
    res = {m: [] for m in calls}
    for _ in range(windows):
        for mode, fn in calls.items():
            with _mode(mode):
                res[mode].append(_window(fn, reps))
    return {m: statistics.median(v) for m, v in res.items()}


class _mode:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        D.set_default_mode(self.mode)

    def __exit__(self, *exc):
        D.set_default_mode('auto')


def forward(reps, emit):
    b, r = 16, 5
    d = bench.make_inputs(b, r, 1234, DEV)
    idx, _ = M.feature_match_index_batched(d['feat_in'], d['feat_ref'], is_norm=True, norm_input=True,
                                           normalize_pixels=True, in_div=r)
    for c, hw in bench.SCALES:
        s = hw // 40
        x, conv_out, w, bias = d[f'x{c}'], d[f'conv_out{c}'], d[f'w{c}'], d[f'b{c}']
        fused = {m: (lambda: D.dynagg_dcn_forward(x, conv_out, idx, s, w, bias, bench.DG)) for m in MODES[:2]}
        for mode, ms in _time_modes(fused, reps).items():
            emit(dict(pass_='forward', entry='fused', C=c, hw=hw, samples=b * r, mode=mode, ms=round(ms, 4)))
        g = torch.Generator(device=DEV).manual_seed(c)
        off = torch.randn(b * r, 2 * bench.DG * 9, hw, hw, generator=g, device=DEV) * 2
        mask = torch.rand(b * r, bench.DG * 9, hw, hw, generator=g, device=DEV)
        xo = x.float().contiguous()
        op = {m: (lambda m=m: D.dcn_forward_raw(xo, off, mask, w, bias, (1, 1), (1, 1), (1, 1), 1, bench.DG, mode=m))
              for m in MODES}
        for mode, ms in _time_modes(op, reps).items():
            emit(dict(pass_='forward', entry='operator', C=c, hw=hw, samples=b * r, mode=mode, ms=round(ms, 4)))
        del off, mask, xo
        torch.cuda.empty_cache()


def backward(reps, emit):
    total = {m: 0.0 for m in MODES}
    for b, c, hw in TRAIN_SHAPES:
        g = torch.Generator(device=DEV).manual_seed(b + c)
        x = torch.randn(b, c, hw, hw, generator=g, device=DEV)
        off = torch.randn(b, 2 * 8 * 9, hw, hw, generator=g, device=DEV) * 2
        mask = torch.rand(b, 8 * 9, hw, hw, generator=g, device=DEV)
        w = torch.randn(c, c, 3, 3, generator=g, device=DEV) * (c * 9) ** -0.5
        go = torch.randn(b, c, hw, hw, generator=g, device=DEV)
        fn = (lambda: D.dcn_backward_raw(x, off, mask, w, go, (1, 1), (1, 1), (1, 1), 1, 8, True))
        times = _time_modes({m: fn for m in MODES}, reps)
        for mode, ms in times.items():
            total[mode] += ms
            emit(dict(pass_='backward', B=b, C=c, hw=hw, mode=mode, ms=round(ms, 4)))
        del x, off, mask, w, go
        torch.cuda.empty_cache()
    for mode, ms in total.items():
        emit(dict(pass_='backward', shape='training step (sum of the three)', mode=mode, ms=round(ms, 4)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n\n')[0])
    ap.add_argument('--reps', type=int, default=10, help='calls per timed window')
    ap.add_argument('--out', help='also append the JSON lines to this file')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('dcn_x3_bench: needs a CUDA device (these are device times)')
    out = open(args.out, 'a') if args.out else None

    def emit(rec):
        rec = {('pass' if k == 'pass_' else k): v for k, v in rec.items()}
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + '\n')
            out.flush()
    emit(_gpu_info())
    forward(args.reps, emit)
    backward(max(1, args.reps // 2), emit)


if __name__ == '__main__':
    main()
