"""
Drop-in for `timbre_trap.framework.objectives` (reference: timbre_trap/framework/objectives.py:1-104): the three
objectives with the reference's signatures, computed by the deterministic reduction kernels of csrc/loss_kernels.cu.
Each is a torch.autograd.Function: with grad mode on and an argument that requires grad, `backward()` reaches both arguments
through the gradient kernels of csrc/train_kernels.cu (tt_sum_sq_diff_bwd, tt_transcription_loss_bwd).  The loss step
(framework/train.py) uses the same Functions.
"""

import torch

from .. import _lib

__all__ = ['compute_reconstruction_loss', 'compute_transcription_loss', 'compute_consistency_loss']


def _same_order(a, b):
    """Two (B, C, F, T) tensors as flat fp32 buffers in one common memory order (free for the kernels' own outputs), and whether
    that order is (B, F, T, C)."""
    a = a.detach().float()
    b = b.detach().float()
    if a.dim() == 4 and a.stride() == b.stride() and a.permute(0, 2, 3, 1).is_contiguous():
        return a.permute(0, 2, 3, 1), b.permute(0, 2, 3, 1), True
    return a.contiguous(), b.contiguous(), False


def _scratch(device):
    return torch.empty(_lib.lib().tt_loss_scratch_floats(), dtype=torch.float32, device=device)


class _SqDiffFn(torch.autograd.Function):
    """scale * sum((a - b)^2) over two tensors of one shape in any memory order (tt_sum_sq_diff); gradients to both in that order
    (tt_sum_sq_diff_bwd), handed back in the shape of the arguments."""

    @staticmethod
    def forward(ctx, a, b, scale):
        x, y, channels_last = _same_order(a, b)
        out = torch.empty((), dtype=torch.float32, device=x.device)
        _lib.launch('tt_sum_sq_diff', x, y, x.numel(), scale, out, _scratch(x.device))
        ctx.save_for_backward(x, y)
        ctx.meta = (scale, channels_last)
        return out

    @staticmethod
    def backward(ctx, gout):
        x, y = ctx.saved_tensors
        scale, channels_last = ctx.meta
        ga = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gb = torch.empty_like(y) if ctx.needs_input_grad[1] else None
        if ga is None and gb is None:
            return None, None, None
        _lib.launch('tt_sum_sq_diff_bwd', x, y, gout.float().contiguous(), scale, ga, gb, x.numel())
        if channels_last:
            ga, gb = [None if g is None else g.permute(0, 3, 1, 2) for g in (ga, gb)]
        return ga, gb, None


def _sum_sq_diff(a, b, frames):
    """sum((a - b)^2) / frames through _SqDiffFn: the reconstruction / consistency loss of tensors in any layout (the loss step
    passes interleaved pairs (B, F, T, 2) as they are)."""
    return _SqDiffFn.apply(a, b, 1.0 / frames)


class _TrnLossFn(torch.autograd.Function):
    """The transcription loss of two (B, F, T) tensors (tt_transcription_loss); gradients to the estimate and / or the target in one
    pass (tt_transcription_loss_bwd)."""

    @staticmethod
    def forward(ctx, estimate, target, weight_positive_class):
        e = estimate.detach().float().contiguous()
        g = target.detach().float().contiguous()
        B, F, T = e.shape
        out = torch.empty((), dtype=torch.float32, device=e.device)
        _lib.launch('tt_transcription_loss', e, g, B, F, T, int(bool(weight_positive_class)), out, _scratch(e.device))
        ctx.save_for_backward(e, g)
        ctx.weighted = int(bool(weight_positive_class))
        return out

    @staticmethod
    def backward(ctx, gout):
        e, g = ctx.saved_tensors
        ge = torch.empty_like(e) if ctx.needs_input_grad[0] else None
        gg = torch.empty_like(g) if ctx.needs_input_grad[1] else None
        if ge is None and gg is None:
            return None, None, None
        B, F, T = e.shape
        _lib.launch('tt_transcription_loss_bwd', e, g, gout.float().contiguous(), B, F, T, ctx.weighted, ge, gg)
        return ge, gg, None


def compute_reconstruction_loss(reconstructed, target):
    """objectives.py:11-33: squared error summed over (C, F), averaged over (B, T).  Differentiable in both arguments."""
    _lib.require_cuda(reconstructed, 'reconstructed')
    _lib.require_cuda(target, 'target')
    if reconstructed.shape != target.shape:
        raise ValueError(f'shape mismatch {tuple(reconstructed.shape)} vs {tuple(target.shape)}')
    return _sum_sq_diff(reconstructed, target, reconstructed.size(0) * reconstructed.size(-1))


def compute_transcription_loss(estimate, target, weight_positive_class=False):
    """objectives.py:36-74.  Differentiable in both arguments (the target also through the positive-class weight)."""
    _lib.require_cuda(estimate, 'estimate')
    _lib.require_cuda(target, 'target')
    if estimate.shape != target.shape or estimate.dim() != 3:
        raise ValueError('estimate and target must both be (B, F, T)')
    return _TrnLossFn.apply(estimate, target, weight_positive_class)


def compute_consistency_loss(spectral_coefficients, transcription_coefficients, target):
    """objectives.py:77-104.  Differentiable in all three arguments."""
    return (compute_reconstruction_loss(spectral_coefficients, target),
            compute_reconstruction_loss(transcription_coefficients, target))
