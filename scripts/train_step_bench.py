"""Times the loss step of BASELINE.json configs[3] (batch 8 x 9 s per GPU) and checks data-parallel gradients when run under torchrun.
Usage: train_step_bench.py [batch] [steps] [base|film|mag|magdb] [trainstep|api]
  variant: the model class to train (default base = TimbreTrap)
  mode:    trainstep (default) - framework.train.TrainStep: one CQT, the native clip + AdamW over one flat bucket;
           api - the reference's loop body (experiments/train.py:393-500) on the public API: model.train(), model(audio, consistency=True),
           to_activations, the three compute_*_loss functions, backward(), clip_grad_norm_(..., 10) and torch.optim.AdamW(lr=1e-3).
           One GPU only."""
import os, sys, time, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist
from timbre_trap_b200.framework import (TimbreTrap, TimbreTrapFiLM, TimbreTrapMag, TimbreTrapMagDB, compute_consistency_loss,
                                        compute_reconstruction_loss, compute_transcription_loss)
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
mode = sys.argv[4] if len(sys.argv) > 4 else 'trainstep'
classes = dict(base=TimbreTrap, film=TimbreTrapFiLM, mag=TimbreTrapMag, magdb=TimbreTrapMagDB)
if variant not in classes:
    sys.exit(f'unknown variant {variant!r}: one of {", ".join(classes)}')
if mode not in ('trainstep', 'api'):
    sys.exit(f'unknown mode {mode!r}: trainstep or api')
if mode == 'api' and world > 1:
    sys.exit('api mode runs on one GPU: data-parallel training is TrainStep\'s (its gradient bucket is all-reduced over NCCL)')
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


def reference_target(model, audio):
    """The reconstruction target: the reference's model.sliCQ(audio) (train.py:404) for TimbreTrap / TimbreTrapFiLM; for the magnitude
    variants their own one-channel encoder input, as TrainStep uses it."""
    coefficients = model.sliCQ(audio)
    if variant in ('base', 'film'):
        return coefficients
    mag = model.sliCQ.to_magnitude(coefficients)
    return (model.sliCQ.to_decibels(mag) if variant == 'magdb' else mag).unsqueeze(1)


class ApiStep:
    """experiments/train.py:393-500 on the public API, with torch's optimizer and clipping."""

    def __init__(self, model):
        self.model = model.train()
        self.opt = torch.optim.AdamW(model.parameters(), lr=1e-3)

    def step(self, audio, gt):
        n = gt.size(0)
        target = reference_target(self.model, audio)
        rec, _, trn, trn_rec, trn_scr, _ = self.model(audio, consistency=True)
        act = self.model.to_activations(trn)
        out = dict(reconstruction=compute_reconstruction_loss(rec, target), transcription=compute_transcription_loss(act[:n], gt, True))
        out['consistency_spectral'], out['consistency_score'] = compute_consistency_loss(trn_rec[:n], trn_scr[:n], trn[:n])
        out['total'] = out['reconstruction'] + out['transcription'] + out['consistency_spectral'] + out['consistency_score']
        self.opt.zero_grad()
        out['total'].backward()
        norm = torch.nn.utils.clip_grad_norm_(self.model.parameters(), 10)
        self.opt.step()
        res = {k: v.detach() for k, v in out.items()}
        res['grad_norm'] = norm
        return res


ts = TrainStep(model, group=group) if mode == 'trainstep' else ApiStep(model)

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
    print(json.dumps(dict(workload='loss step, %s model, batch %d x 9 s per GPU' % (variant, B), mode=mode, n_gpus=world, ms_per_step=ms,
                          audio_s_per_s=world * B * 9 / (ms * 1e-3), losses={k: float(v) for k, v in res.items()},
                          peak_mem_gb=torch.cuda.max_memory_allocated() / 1e9)))
if world > 1: dist.destroy_process_group()
