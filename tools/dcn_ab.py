"""A/B timing of the fused DynAgg + DCNv2 launches on bench.py's config-2 inputs, per scale.

    MREFSR_LIB=<variant .so> python tools/dcn_ab.py [tag]

Prints one JSON line per (flow kind, scale): per-launch device time of dcn_tc_split_kernel (CUDA events recorded
inside the library).  Flow kinds: 'bench' = the arg-max maps of bench.py's synthetic references (3 translated, 2 independent
per image), 'coherent' = every reference a translation, 'random' = uniformly random arg-max maps.
"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import mrefsr_b200 as M  # noqa: E402
from mrefsr_b200 import _lib  # noqa: E402
from mrefsr_b200.dcn import dynagg_dcn_forward  # noqa: E402

DEV = 'cuda:0'


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else ''
    b, r = 16, 5
    d = bench.make_inputs(b, r, 1234, DEV)
    idx, _ = M.feature_match_index_batched(d['feat_in'], d['feat_ref'], is_norm=True, norm_input=True,
                                           normalize_pixels=True, in_div=r)
    g = torch.Generator().manual_seed(7)
    ys, xs = torch.meshgrid(torch.arange(38), torch.arange(38), indexing='ij')
    coh = []
    for k in range(b * r):
        dy, dx = int(torch.randint(-6, 7, (1,), generator=g)), int(torch.randint(-6, 7, (1,), generator=g))
        coh.append((ys + dy).clamp(0, 37) * 38 + (xs + dx).clamp(0, 37))
    flows = {'bench': idx, 'coherent': torch.stack(coh).to(DEV),
             'random': torch.randint(0, 38 * 38, (b * r, 38, 38), generator=g).to(DEV)}
    outs = {}
    for kind, mi in flows.items():
        total = 0.0
        for c, hw in bench.SCALES:
            args = (d[f'x{c}'], d[f'conv_out{c}'], mi, hw // 40, d[f'w{c}'], d[f'b{c}'], bench.DG)
            for _ in range(2):
                y = dynagg_dcn_forward(*args)
            torch.cuda.synchronize()
            _lib.timing_enable(True)
            _lib.timing_read()
            for _ in range(5):
                y = dynagg_dcn_forward(*args)
            t = _lib.timing_read()
            _lib.timing_enable(False)
            ms = t['dcn_fwd'][0] / max(1, t['dcn_fwd'][1])
            total += ms
            outs[(kind, c)] = y
            print(json.dumps(dict(tag=tag, flow=kind, C=c, hw=hw, ms=round(ms, 4), aux_ms=round(t['dcn_aux'][0] / max(1, t['dcn_aux'][1]), 4),
                                  checksum=float(y.double().sum()))), flush=True)
        print(json.dumps(dict(tag=tag, flow=kind, total_ms=round(total, 4))), flush=True)


if __name__ == '__main__':
    main()
