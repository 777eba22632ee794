"""BASELINE config 5: stage-3 restoration training step (L1 pixel loss, Adam on net_g only, DDP when launched with
torchrun), 5 refs @160^2, through this repo's DynAgg / DCNv2 / MRAPAFusion autograd Functions (reference operator
boundaries: materialised pre-offsets, modulated_deform_conv backward for offset / mask / weight / bias, fusion
backward).  The matcher has no backward (its only consumed output is the integer arg-max, SURVEY.md section 3.2).

  python tools/train_step_bench.py [--batch 4] [--steps 5] [--bf16] [--fused-dynagg]
  python -m torch.distributed.run --nproc-per-node N tools/train_step_bench.py ...
Prints one JSON line on rank 0."""
import argparse
import json
import os
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mrefsr_b200.models import MRefSRPipeline  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument('--batch', type=int, default=4)
ap.add_argument('--refs', type=int, default=5)
ap.add_argument('--steps', type=int, default=5)
ap.add_argument('--hr', type=int, default=160)
ap.add_argument('--channels-last', action='store_true', help='run net_g in torch.channels_last (cuDNN native layout)')
ap.add_argument('--per-reference', action='store_true', help='evaluate the frozen nets once per reference (the reference model structure)')
ap.add_argument('--bf16', action='store_true', help='bf16 autocast for the plain convolutions (hot-path ops stay fp32)')
ap.add_argument('--fused-dynagg', action='store_true',
                help='train on the fused DynAgg path: correspondences(..., as_max_idx=True) -> net_g(lq, max_idx, feats, r), '
                     'offsets / masks built inside the DCN gather in the forward and the backward')
args = ap.parse_args()
if args.fused_dynagg and args.per_reference:
    ap.error('--fused-dynagg takes the batched correspondences (no --per-reference)')

rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
local = int(os.environ.get('LOCAL_RANK', 0))
torch.cuda.set_device(local)
dev = torch.device('cuda', local)
if world > 1:
    dist.init_process_group('nccl', device_id=dev)

torch.manual_seed(10)
pipe = MRefSRPipeline().to(dev)
pipe.net_extractor.eval()
pipe.net_map.eval()
for p in list(pipe.net_extractor.parameters()) + list(pipe.net_map.parameters()):
    p.requires_grad_(False)
net_g = pipe.net_g.train()
if args.channels_last:
    pipe.channels_last_()                    # net_g and the frozen nets in torch.channels_last
# learned offsets start at zero in the reference; give them a little signal so every backward path is exercised
for name in ('small', 'medium', 'large'):
    getattr(net_g.dyn_agg_restore, f'{name}_dyn_agg').conv_offset_mask.weight.data.normal_(0, 1e-3)
model = torch.nn.parallel.DistributedDataParallel(net_g, device_ids=[local]) if world > 1 else net_g
opt = torch.optim.Adam(net_g.parameters(), lr=1e-4)

b, r, H = args.batch, args.refs, args.hr
g = torch.Generator().manual_seed(1234 + rank)
gt = torch.rand(b, 3, H, H, generator=g).to(dev)
lq = torch.nn.functional.interpolate(gt, scale_factor=0.25, mode='bicubic', align_corners=False).clamp(0, 1)
up = torch.nn.functional.interpolate(lq, scale_factor=4, mode='bicubic', align_corners=False).clamp(0, 1)
refs = [torch.rand(b, 3, H, H, generator=g).to(dev) for _ in range(r)]


refs_stacked = torch.stack(refs, 1)                              # [B, R, 3, H, W]


def step():
    if args.per_reference:      # the reference's own structure: one net_extractor / net_map evaluation per reference
        with torch.no_grad():
            feats = pipe.net_extractor(up, refs)
            pres, rfs = [], []
            for f, ref in zip(feats, refs):
                pre, rf = pipe.net_map(f, ref)
                pres.append(pre)
                rfs.append(rf)
        n_refs = None
    else:                       # the same, batched over the references (one extractor / matcher / VGG pass)
        pres, rfs, n_refs = pipe.correspondences(up, refs_stacked, as_max_idx=args.fused_dynagg)
    opt.zero_grad(set_to_none=True)
    x_in = lq.contiguous(memory_format=torch.channels_last) if args.channels_last else lq
    with torch.autocast('cuda', dtype=torch.bfloat16, enabled=args.bf16):
        out = model(x_in, pres, rfs, n_refs)
    loss = torch.nn.functional.l1_loss(out.float(), gt)
    loss.backward()
    opt.step()
    return loss


losses = [float(step()) for _ in range(2)]
torch.cuda.synchronize()
torch.cuda.reset_peak_memory_stats(dev)
if world > 1:
    dist.barrier()
t0 = time.perf_counter()
for _ in range(args.steps):
    losses.append(float(step()))
torch.cuda.synchronize()
dt = torch.tensor([(time.perf_counter() - t0) / args.steps], device=dev, dtype=torch.float64)
if world > 1:
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
grads_ok = all(p.grad is not None and torch.isfinite(p.grad).all() for p in net_g.parameters())
if rank == 0:
    print(json.dumps({'test': 'train_step', 'n_gpus': world, 'batch_per_gpu': b, 'refs': r, 'hr': H, 'bf16_convs': args.bf16,
                      'fused_dynagg': args.fused_dynagg, 'ms_per_step': float(dt) * 1e3,
                      'max_memory_allocated_gb': torch.cuda.max_memory_allocated(dev) / 2 ** 30, 'images_per_s': b * world / float(dt), 'losses': [round(x, 5) for x in losses],
                      'loss_decreasing': losses[-1] < losses[0], 'all_grads_finite': bool(grads_ok)}), flush=True)
if world > 1:
    dist.destroy_process_group()
