"""
The data path's front end and evaluation metric on the device (SURVEY.md section 8f-3 / 8f-4), so that a long clip can go
from decoded samples to model input - and from model output to the reported metrics - without leaving the GPU:

  prepare_audio(audio, fs, sample_rate)        AudioDataset.get_audio after torchaudio.load (datasets/AudioDataset.py:69-77):
                                               mono mix, torchaudio.functional.resample, infinity-norm normalise
  multi_pitch_to_activations(...)              PitchDataset.multi_pitch_to_activations (datasets/PitchDataset.py:233-307)
  signal_distortion_ratio(preds, target)       torchmetrics SignalDistortionRatio as experiments/evaluate.py:51,122-127 uses it

Kernels: csrc/frontend_kernels.cu through the C ABI.  No CPU fallback.
"""

import math

import numpy as np
import torch

from .. import _lib

__all__ = ['prepare_audio', 'sinc_resample_kernel', 'multi_pitch_to_activations', 'signal_distortion_ratio']


def sinc_resample_kernel(orig_freq, new_freq, lowpass_filter_width=6, rolloff=0.99):
    """
    The filter bank of torchaudio.functional.resample (resampling_method 'sinc_interp_hann', the default the reference uses at
    AudioDataset.py:73): for output phase j in [0, new) the taps k in [-width, width + orig) of a Hann-windowed sinc at the
    band edge min(orig, new) * rolloff.  Returns (kernel (new, 2 * width + orig) float32, orig, new, width) with the
    frequencies divided by their gcd.
    """
    if int(orig_freq) != orig_freq or int(new_freq) != new_freq or orig_freq <= 0 or new_freq <= 0:
        raise ValueError('sample rates must be positive integers')
    g = math.gcd(int(orig_freq), int(new_freq))
    orig, new = int(orig_freq) // g, int(new_freq) // g
    base = min(orig, new) * rolloff
    width = math.ceil(lowpass_filter_width * orig / base)
    # float32 arithmetic in torchaudio's order: the reference resamples float32 audio, for which torchaudio builds this table in
    # float32 (the large sinc arguments make that differ from a float64 table at the 1e-5 level - parity means matching it)
    f32 = torch.float32
    idx = torch.arange(-width, width + orig, dtype=f32)[None, :] / orig
    t = torch.arange(0, -new, -1, dtype=f32)[:, None] / new + idx
    t = (t * base).clamp_(-lowpass_filter_width, lowpass_filter_width)
    window = torch.cos(t * math.pi / lowpass_filter_width / 2) ** 2
    t = t * math.pi
    kern = torch.where(t == 0, torch.tensor(1.0, dtype=f32), t.sin() / t) * (window * (base / orig))
    return kern.numpy().astype(np.float32), orig, new, width


_KERNELS = {}


def prepare_audio(audio, fs, sample_rate, normalise=True):
    """
    audio (C, N) fp32 CUDA tensor as torchaudio.load returns it, sampled at `fs` -> (1, N') at `sample_rate`:
    mean over channels, resample, divide by the peak if it is non-zero (AudioDataset.py:71-77).
    """
    _lib.require_cuda(audio, 'audio')
    if audio.dim() != 2:
        raise ValueError(f'audio must be (channels, samples), got {tuple(audio.shape)}')
    audio = audio.detach().float().contiguous()
    C, N = audio.shape
    key = (int(fs), int(sample_rate), audio.device)
    if key not in _KERNELS:
        if int(fs) == int(sample_rate):
            table, orig, new, width = np.ones((1, 1), dtype=np.float32), 1, 1, 0
        else:
            table, orig, new, width = sinc_resample_kernel(fs, sample_rate)
        _KERNELS[key] = (torch.from_numpy(table).to(audio.device), orig, new, width)
    table, orig, new, width = _KERNELS[key]
    n_out = int(math.ceil(new * N / orig))
    out = torch.empty((1, n_out), dtype=torch.float32, device=audio.device)
    peak = torch.empty((), dtype=torch.float32, device=audio.device)
    _lib.launch('tt_resample_mono', audio, C, N, table, orig, new, width, out, n_out, peak)
    if normalise and n_out:
        _lib.launch('tt_scale_by_peak', out, n_out, peak)
    return out


def _gaussian_taps(sigma, truncate=4.0):
    """scipy.ndimage.gaussian_filter1d's kernel: radius int(truncate * sigma + 0.5), exp(-x^2 / (2 sigma^2)), normalised."""
    radius = int(truncate * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1, dtype=np.float64)
    w = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return (w / w.sum()).astype(np.float32), radius


def multi_pitch_to_activations(multi_pitch, midi_freqs, n_bins_blur_decay=2.5, device=None):
    """
    multi_pitch: list (one entry per frame) of arrays of active pitches in Hz, or a dense (T, P) array / tensor padded with zeros;
    midi_freqs (F) ascending.  Returns the (F, T) fp32 activation map on the device (PitchDataset.py:233-307).
    """
    if isinstance(multi_pitch, torch.Tensor):
        dense = multi_pitch.detach().to(torch.float64)
        device = dense.device if device is None else torch.device(device)
    else:
        if isinstance(multi_pitch, np.ndarray) and multi_pitch.ndim == 2:
            host = np.asarray(multi_pitch, dtype=np.float64)
        else:
            T = len(multi_pitch)
            P = max([len(p) for p in multi_pitch], default=0)
            host = np.zeros((T, max(P, 1)), dtype=np.float64)
            for i, p in enumerate(multi_pitch):
                host[i, :len(p)] = np.asarray(p, dtype=np.float64)
        if device is None:
            raise ValueError('pass device= when multi_pitch is not a tensor')
        dense = torch.from_numpy(host)
    device = torch.device(device)
    if device.type != 'cuda':
        raise _lib.TimbreTrapB200Error('multi_pitch_to_activations runs on a CUDA device (the CPU oracle lives in oracle/)')
    dense = dense.to(device).contiguous()
    T, P = dense.shape
    freqs = torch.as_tensor(np.asarray(midi_freqs, dtype=np.float64), device=device).contiguous()
    F = freqs.numel()
    if n_bins_blur_decay:
        taps, radius = _gaussian_taps((2 * n_bins_blur_decay) / 5)
    else:
        taps, radius = np.ones(1, dtype=np.float32), 0
    blur = torch.from_numpy(taps).to(device)
    act = torch.empty((F, T), dtype=torch.float32, device=device)
    scratch = torch.empty(1, dtype=torch.float32, device=device)
    _lib.launch('tt_rasterise_pitches', dense, T, P, freqs, F, blur, radius, act, scratch)
    return act


def signal_distortion_ratio(preds, target, filter_length=512, zero_mean=False, load_diag=None):
    """
    SDR in dB per item, (..., N) -> (...): the definition torchmetrics' SignalDistortionRatio implements (the reference builds it at
    experiments/evaluate.py:51 with default arguments and calls it on (synth, audio) at :125): both signals scaled to unit norm,
    the length-`filter_length` distortion filter is the solution of the Toeplitz normal equations R h = b (R from the target's
    auto-correlation, b its cross-correlation with the estimate), coherence = b . h, SDR = 10 log10(coh / (1 - coh)).
    The O(N * filter_length) correlations run in fp64 in tt_sdr_correlations; the 512 x 512 solve is a library call.
    torchmetrics is not in this image: the restatement is checked against a dense numpy evaluation of the same definition.
    """
    _lib.require_cuda(preds, 'preds')
    if preds.shape != target.shape:
        raise ValueError('preds and target must have the same shape')
    shape = preds.shape[:-1]
    n = preds.size(-1)
    p = preds.detach().float().reshape(-1, n)
    t = target.detach().float().reshape(-1, n)
    if zero_mean:
        p = p - p.mean(dim=-1, keepdim=True)
        t = t - t.mean(dim=-1, keepdim=True)
    p, t = p.contiguous(), t.contiguous()
    B = p.size(0)
    r0 = torch.empty((B, filter_length), dtype=torch.float64, device=p.device)
    b = torch.empty_like(r0)
    norms = torch.empty((B, 2), dtype=torch.float64, device=p.device)
    _lib.launch('tt_sdr_correlations', t, p, B, n, filter_length, r0, b, norms)
    nt = norms[:, 0].sqrt().clamp(min=1e-6)
    npred = norms[:, 1].sqrt().clamp(min=1e-6)
    r0 = r0 / (nt * nt).unsqueeze(-1)
    b = b / (nt * npred).unsqueeze(-1)
    if load_diag is not None:
        r0[:, 0] += load_diag
    idx = (torch.arange(filter_length, device=p.device)[:, None] - torch.arange(filter_length, device=p.device)[None, :]).abs()
    sol = torch.linalg.solve(r0[:, idx], b.unsqueeze(-1)).squeeze(-1)
    coh = (b * sol).sum(-1)
    return (10.0 * torch.log10(coh / (1 - coh))).to(preds.dtype).reshape(shape)
