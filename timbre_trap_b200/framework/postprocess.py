"""
Evaluation post-processing on the device - the step that follows `TimbreTrap.transcribe` in the reference's evaluation
(experiments/evaluate.py:98-116), SURVEY.md section 8f-1.  Same names and argument meaning as the reference's numpy functions,
but on CUDA tensors (CPU tensors raise: there is no fallback):

  filter_non_peaks(activations)                       timbre_trap/utils/processing.py:66-98
  threshold(activations, t=0.5)                       timbre_trap/utils/processing.py:101-124
  activations_to_binary(activations, ...)             PitchDataset.activations_to_multi_pitch (datasets/PitchDataset.py:309-349) up
                                                      to the binary map (+ the bin mask of evaluate.py:48), one fused kernel
  multipitch_counts / multipitch_scores               mir_eval.multipitch precision / recall / f1 (utils/experiments.py:354-396) for
                                                      estimates and references on a common frame grid
"""

import sys

import torch

from .. import _lib

__all__ = ['filter_non_peaks', 'threshold', 'activations_to_binary', 'multipitch_counts', 'multipitch_scores']


def _as_bft(x, name):
    _lib.require_cuda(x, name)
    if x.dim() < 2:
        raise ValueError(f'{name} must have shape (..., F, T), got {tuple(x.shape)}')
    return x.reshape(-1, x.size(-2), x.size(-1))


def filter_non_peaks(activations):
    """(..., F, T) -> same shape fp32: values that are strict local maxima along the frequency axis (zeros beyond the edges), else 0."""
    a = _as_bft(activations, 'activations').to(torch.float32).contiguous()
    out = torch.empty_like(a)
    B, F, T = a.shape
    if a.numel() == 0:
        return out.reshape(activations.shape)
    _lib.launch('tt_filter_non_peaks', a, out, B, F, T)
    return out.reshape(activations.shape)


def activations_to_binary(activations, t=0.5, peaks_only=False, bin_lo=0, bin_hi=None):
    """(..., F, T) activations -> uint8 {0,1}: optional peak picking, `>= t`, bins outside [bin_lo, bin_hi) cleared."""
    a = _as_bft(activations, 'activations').to(torch.float32).contiguous()
    B, F, T = a.shape
    out = torch.empty((B, F, T), dtype=torch.uint8, device=a.device)
    if a.numel() == 0:
        return out.reshape(activations.shape)
    _lib.launch('tt_peak_threshold', a, out, B, F, T, float(t), int(peaks_only), int(bin_lo), int(F if bin_hi is None else bin_hi))
    return out.reshape(activations.shape)


def threshold(activations, t=0.5):
    """(..., F, T) -> fp32 {0., 1.} like the reference's `threshold` (processing.py:101-124)."""
    return activations_to_binary(activations, t).to(torch.float32)


def multipitch_counts(est, ref, tolerance_bins):
    """est, ref: (..., F, T) binary maps on the same frame grid -> int64 (B, 3): true positives, estimated, reference per item."""
    e = _as_bft(est, 'est').to(torch.uint8).contiguous()
    r = _as_bft(ref, 'ref').to(torch.uint8).contiguous()
    if e.shape != r.shape:
        raise ValueError(f'est {tuple(e.shape)} and ref {tuple(r.shape)} must have the same shape')
    B, F, T = e.shape
    counts = torch.zeros((B, 3), dtype=torch.int64, device=e.device)
    if e.numel() == 0:
        return counts
    _lib.launch('tt_multipitch_counts', e, r, B, F, T, int(tolerance_bins), counts)
    return counts


def multipitch_scores(est, ref, tolerance_bins):
    """Precision, recall and f1 over all items (one host read of three integers), as utils/experiments.py:375-392 reports them."""
    tp, n_est, n_ref = (int(v) for v in multipitch_counts(est, ref, tolerance_bins).sum(0).tolist())
    p = tp / n_est if n_est else 0.0
    r = tp / n_ref if n_ref else 0.0
    return {'precision': p, 'recall': r, 'f1-score': 2 * p * r / (p + r + sys.float_info.epsilon)}
