"""Ablation timing of the DCN forward kernel (variant build with -DMREFSR_DCN_DEBUG; MREFSR_DCN_DBG bit mask, see
csrc/dcn_tc.cu).  Results are wrong by design; only the time matters.  One JSON line per scale."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from mrefsr_b200 import _lib  # noqa: E402
from mrefsr_b200.dcn import dynagg_dcn_forward  # noqa: E402

DEV = 'cuda:0'
tag = sys.argv[1] if len(sys.argv) > 1 else ''
scales = [int(a) for a in sys.argv[2:]] or [64]
d = bench.make_inputs(16, 5, 1234, DEV)
ys, xs = torch.meshgrid(torch.arange(38), torch.arange(38), indexing='ij')
mi = torch.stack([(ys + 2).clamp(0, 37) * 38 + (xs - 3).clamp(0, 37)] * 80).to(DEV)
for c, hw in bench.SCALES:
    if c not in scales:
        continue
    args = (d[f'x{c}'], d[f'conv_out{c}'], mi, hw // 40, d[f'w{c}'], d[f'b{c}'], bench.DG)
    for _ in range(2):
        dynagg_dcn_forward(*args)
    torch.cuda.synchronize()
    _lib.timing_enable(True)
    _lib.timing_read()
    for _ in range(5):
        dynagg_dcn_forward(*args)
    t = _lib.timing_read()
    _lib.timing_enable(False)
    print(json.dumps(dict(tag=tag, dbg=os.environ.get('MREFSR_DCN_DBG', '0'), C=c,
                          ms=round(t['dcn_fwd'][0] / max(1, t['dcn_fwd'][1]), 4))), flush=True)
