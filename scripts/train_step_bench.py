"""Times the loss step of BASELINE.json configs[3] (batch 8 x 9 s per GPU) and checks data-parallel gradients when run under torchrun.
Usage: train_step_bench.py [batch] [steps] [base|film|mag|magdb] - the model class to train (default base = TimbreTrap)."""
import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from timbre_trap_b200.framework import TimbreTrap, TimbreTrapFiLM, TimbreTrapMag, TimbreTrapMagDB
from timbre_trap_b200.framework.train import TrainStep

rank, world, local = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1)), int(os.environ.get('LOCAL_RANK', 0))
torch.cuda.set_device(local)
group = None
if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    group = dist.group.WORLD
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
variant = sys.argv[3] if len(sys.argv) > 3 else 'base'
classes = dict(base=TimbreTrap, film=TimbreTrapFiLM, mag=TimbreTrapMag, magdb=TimbreTrapMagDB)
if variant not in classes:
    sys.exit(f'unknown variant {variant!r}: one of {", ".join(classes)}')
torch.manual_seed(0)
model = classes[variant](22050, 9, 60, 3, latent_size=128, model_complexity=2).cuda()
g = torch.Generator().manual_seed(100 + rank)
audio = (torch.rand((B, 1, 3 * 66150), generator=g) * 2 - 1).cuda()
gt = torch.zeros((B, 540, 3072))
rng = np.random.default_rng(rank)
for b in range(B):
    for k in rng.integers(60, 480, size=4):
        gt[b, k] = 1.0
        gt[b, k - 1] = gt[b, k + 1] = 0.6
gt = gt.cuda()
ts = TrainStep(model, group=group)

if world > 1:
    # data-parallel check: the all-reduced gradient equals the mean of the per-rank gradients
    out = ts.losses(audio, gt)
    for p in ts.params: p.grad = None
    out['total'].backward()
    local_flat = torch.cat([p.grad.reshape(-1) for p in ts.params]).clone()
    gathered = [torch.empty_like(local_flat) for _ in range(world)]
    dist.all_gather(gathered, local_flat)
    want = torch.stack(gathered).mean(0)
    ts.backward(ts.losses(audio, gt)['total'])
    got = torch.cat([p.grad.reshape(-1) for p in ts.params])
    err = float((got - want).norm() / want.norm())
    if rank == 0: print('ddp gradient check: rel err vs mean of per-rank gradients', err, 'bucket bytes', got.numel() * 4)
    assert err < 1e-3

for _ in range(3): ts.step(audio, gt)
torch.cuda.synchronize()
if world > 1: dist.barrier()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(steps): res = ts.step(audio, gt)
b.record(); torch.cuda.synchronize()
ms = a.elapsed_time(b) / steps
if world > 1:
    t = torch.tensor([ms], device='cuda'); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t)
if rank == 0:
    print(json.dumps(dict(workload='loss step, %s model, batch %d x 9 s per GPU' % (variant, B), n_gpus=world, ms_per_step=ms,
                          audio_s_per_s=world * B * 9 / (ms * 1e-3), losses={k: float(v) for k, v in res.items()},
                          peak_mem_gb=torch.cuda.max_memory_allocated() / 1e9)))
if world > 1: dist.destroy_process_group()
