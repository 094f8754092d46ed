"""
The reference's loss step (reference: experiments/train.py:393-500) on the CUDA kernels.

  compute_step_losses(model, audio, ground_truth)   forward half only (no graph): evaluation / validation losses
  TrainStep(model, ...).step(audio, ground_truth)   the whole step: CQT target (once), forward with consistency, the four
                                                    losses, backward, gradient all-reduce (NCCL, when a process group is
                                                    given), clip_grad_norm_(10), AdamW

The forward is the model's own (TimbreTrap._passes); with gradients every layer runs as a torch.autograd.Function whose forward is the
inference kernel and whose backward stays in the bf16 inference layouts (framework/layer_grads.py); clip and AdamW have kernels of
their own (csrc/train_kernels.cu).  PyTorch's autograd engine only walks the graph and accumulates `.grad`; there is no cuDNN / ATen
compute on the path.
The reference's own loop body on the public API (model.train(), model(audio, consistency=True), to_activations, the compute_*_loss
functions, backward(), any torch optimizer) runs the same Functions; see INTEGRATION.md section 4.
Differences to the reference that do not change values: the CQT target is computed once (the reference computes it twice,
train.py:404 and modules.py:366 -> :88); no `.item()` host syncs inside the step; activation gradients travel in bf16 between
layers (the reference runs the forward under fp16 autocast).
"""

import torch

from .. import _lib
from . import packing as P  # noqa: F401
from .layer_grads import _ActivationsFn, _Channel0ActivationsFn, _p, _s
from .objectives import _sum_sq_diff, _TrnLossFn
# the weight-gradient and edge-kernel wrappers, where code written against the earlier layout of this module reaches them
from .layer_grads import _channel0_bwd, _film_convin_grads, _wgrad_lat, _wgrad_same, _wgrad_updown  # noqa: F401
from .packing import _PackedCache

__all__ = ['compute_step_losses', 'TrainStep', 'allreduce_mean_gradients']


def _step_losses(model, audio, ground_truth, mult, late_start, grad):
    """The losses of compute_step_losses / TrainStep.losses; `grad`: the model's layers through their autograd Functions.  The
    transcription loss is formed before the consistency pass, so that autograd adds up the transcription's gradients in one order."""
    with torch.no_grad():
        coeffs = model._features(audio)                                     # the reconstruction target (see TrainStep), computed once
    rec, trn, _ = model._passes(coeffs, grad)
    mode = model.ACTIVATIONS_MODE
    act = _ActivationsFn.apply(trn) if mode is None else _Channel0ActivationsFn.apply(trn, mode)
    n = ground_truth.size(0)
    frames = rec.size(0) * rec.size(2)
    out = dict(reconstruction=_sum_sq_diff(rec, coeffs, frames),
               transcription=_TrnLossFn.apply(act[:n].contiguous(), ground_truth.float().contiguous(), True))
    total = mult['reconstruction'] * out['reconstruction']
    if mult['consistency']:
        trn_rec, trn_scr, _ = model._passes(trn, grad)
        tgt = trn[:n].contiguous()
        out['consistency_spectral'] = _sum_sq_diff(trn_rec[:n].contiguous(), tgt, n * tgt.size(2))
        out['consistency_score'] = _sum_sq_diff(trn_scr[:n].contiguous(), tgt, n * tgt.size(2))
    if not late_start:
        total = total + mult['transcription'] * out['transcription']
        if mult['consistency']:
            total = total + mult['consistency'] * (out['consistency_spectral'] + out['consistency_score'])
    out['total'] = total
    return out


def compute_step_losses(model, audio, ground_truth, multipliers=None, late_start=False):
    """
    audio (B, 1, n*L) on the GPU, ground_truth (B_mpe, F, T) with B_mpe <= B (train.py:393-394, 429).
    Returns a dict of 0-dim tensors: reconstruction, transcription, consistency_spectral, consistency_score, total
    (train.py:424-458; `late_start` = True reproduces the epochs before n_epochs_late_start, where only the reconstruction
    term enters the total).  The model variants are scored as TrainStep optimises them: the reconstruction target is the variant's
    own encoder input (model._features), the magnitude variants' outputs pass through their head as pairs (h, 0).
    """
    mult = dict(reconstruction=1, transcription=1, consistency=1)
    mult.update(multipliers or {})
    with torch.no_grad():
        return _step_losses(model, audio, ground_truth, mult, late_start, grad=False)


def allreduce_mean_gradients(params, group, flat=None):
    """Replicas with equal per-rank batches: the mean over ranks of the per-rank gradients is the gradient of the reference's
    global `.mean()` losses (objectives.py:31,72).  One flat bucket (base model: 614,490 fp32 = 2.46 MB), one all-reduce (NCCL on
    the GPU path; any backend works - tests/test_sharding_gloo.py runs it over gloo).  `flat`: the bucket the `.grad` tensors are
    views of (TrainStep) - reduced in place; without it the gradients are gathered into a bucket and copied back."""
    import torch.distributed as dist
    if flat is not None:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat /= dist.get_world_size(group)
        return
    flat = torch.cat([p.grad.reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat /= dist.get_world_size(group)
    off = 0
    for p in params:
        p.grad.copy_(flat[off:off + p.numel()].view_as(p))
        off += p.numel()


class TrainStep:
    """
    One optimisation step of experiments/train.py:393-500 for TimbreTrap, TimbreTrapFiLM, TimbreTrapMag or TimbreTrapMagDB (each with
    or without skip connections): losses as in compute_step_losses, backward, optional NCCL all-reduce of one flat gradient bucket
    (mean over ranks), clip_grad_norm_(max_norm) and AdamW (torch defaults: betas (0.9, 0.999), eps 1e-8, weight_decay 1e-2;
    train.py:334).

    The reconstruction target is the variant's own encoder input, `model._features(audio)`, without gradient: the CQT coefficients
    for TimbreTrap and TimbreTrapFiLM, |c| for TimbreTrapMag and to_decibels(|c|) for TimbreTrapMagDB.  (The reference's loss step
    takes its target from model.sliCQ(audio), train.py:404, whose two channels cannot be compared with the one-channel output of the
    magnitude variants.)  Their one-channel tensors run as pairs (x, 0); the loss over such pairs is the one-channel loss.
    """

    def __init__(self, model, lr=1e-3, max_norm=10.0, multipliers=None, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, group=None):
        self.model = model
        self.params = [p for p in model.parameters()]
        self.lr, self.max_norm, self.betas, self.eps, self.wd = lr, max_norm, betas, eps, weight_decay
        self.mult = dict(reconstruction=1, transcription=1, consistency=1)
        self.mult.update(multipliers or {})
        self.group = group
        self.t = 0
        # ONE flat fp32 bucket each for parameters, gradients and the two AdamW moments: every parameter (and its .grad) is a view
        # into it, so autograd accumulates straight into the bucket, the NCCL all-reduce runs on it in place, and clip + AdamW are
        # two launches over 614,490 floats instead of 2 x 120 (train.py:493-496)
        dev = self.params[0].device
        total = sum(p.numel() for p in self.params)
        self.flat_p = torch.empty(total, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(total, dtype=torch.float32, device=dev)
        self.flat_m = torch.zeros(total, dtype=torch.float32, device=dev)
        self.flat_v = torch.zeros(total, dtype=torch.float32, device=dev)
        self._grad_views = []
        off = 0
        with torch.no_grad():
            for p in self.params:
                n = p.numel()
                self.flat_p[off:off + n].copy_(p.detach().reshape(-1))
                p.data = self.flat_p[off:off + n].view(p.shape)
                self._grad_views.append(self.flat_g[off:off + n].view(p.shape))
                off += n
        _PackedCache.epoch += 1

    def losses(self, audio, ground_truth, late_start=False):
        """The four losses and their total, with the autograd graph attached."""
        return _step_losses(self.model, audio, ground_truth, self.mult, late_start, grad=True)

    def backward(self, total):
        self.flat_g.zero_()
        for p, g in zip(self.params, self._grad_views):
            p.grad = g                                  # autograd accumulates in place: the gradients land in the flat bucket
        total.backward()
        if self.group is not None:
            self._sync_grad_views()
            allreduce_mean_gradients(self.params, self.group, flat=self.flat_g)

    def _sync_grad_views(self):
        """Gradients that were assigned from outside (p.grad = tensor) instead of accumulated by backward(): copy into the bucket."""
        for p, g in zip(self.params, self._grad_views):
            if p.grad is None:
                g.zero_()
            elif p.grad.data_ptr() != g.data_ptr():
                g.copy_(p.grad)
                p.grad = g

    def optimizer_step(self):
        self.t += 1
        self._sync_grad_views()
        acc = torch.zeros((), dtype=torch.float64, device=self.flat_p.device)
        lib = _lib.lib()
        n = self.flat_p.numel()
        _lib.check(lib.tt_grad_sumsq(_p(self.flat_g), n, _p(acc), _s(self.flat_g)))
        _lib.check(lib.tt_adamw_step(_p(self.flat_p), _p(self.flat_g), _p(self.flat_m), _p(self.flat_v), n, _p(acc), self.max_norm, self.lr,
                                     self.betas[0], self.betas[1], self.eps, self.wd, self.t, _s(self.flat_p)))
        _PackedCache.epoch += 1                                                  # weights changed behind torch's back: repack lazily
        return acc.sqrt()

    def step(self, audio, ground_truth, late_start=False):
        """Returns the losses (detached 0-dim tensors) and the pre-clip gradient norm."""
        out = self.losses(audio, ground_truth, late_start)
        self.backward(out['total'])
        norm = self.optimizer_step()
        res = {k: v.detach() for k, v in out.items()}
        res['grad_norm'] = norm
        return res
