"""
Drop-in for `timbre_trap.framework.CQT` (reference: timbre_trap/framework/cqtwrapper.py:10-308,
which subclasses the un-vendored `cqt_pytorch.CQT`).  Same constructor, attributes and methods;
the arithmetic runs in the sm_100a kernels of csrc/cqt_kernels.cu through the C ABI.

Memory contract (same as the reference): `forward` returns a (B, 2, F, T) *view* of an
interleaved (B, F, T, 2) buffer (cqtwrapper.py:91-95), i.e. channels-last memory, which is
what the kernels write and what the conv stack and `decode` read without any re-layout.
"""

import ctypes
import math

import numpy as np
import torch

from .. import _lib
from ..nsgt_tables import FilterBank

__all__ = ['CQT']


def _i32(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))


def _f32(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


class _Plan:
    """Owns one tt_cqt_plan (device tables + scratch) on one device."""

    def __init__(self, bank, device, max_blocks, lanes):
        self.device = device
        self.handle = ctypes.c_void_p()
        with torch.cuda.device(device):
            _lib.check(_lib.lib().tt_cqt_plan_create(
                ctypes.byref(self.handle), bank.block_length, bank.n_bins, bank.max_window_length,
                _i32(bank.start), _i32(bank.length), _i32(bank.first), _i32(bank.offset),
                _f32(bank.win), _f32(bank.dual), bank.n_taps, max_blocks))
            _lib.check(_lib.lib().tt_cqt_plan_set_lanes(self.handle, lanes))

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().tt_cqt_plan_destroy(self.handle)
        except Exception:
            pass


class CQT(torch.nn.Module):
    """
    Invertible NSGT-based constant-Q transform over fixed-length blocks (cqtwrapper.py:10).
    """

    # blocks per kernel group: bounds the plan's scratch (two complex half-spectra per block)
    BLOCKS_PER_LAUNCH = 64
    # internal streams the groups rotate over (front-end FFT kernels of one group overlap the per-bin kernel of another)
    LANES = 2

    def __init__(self, n_octaves, bins_per_octave, sample_rate, secs_per_block):
        """Same signature as the reference (cqtwrapper.py:15-48)."""
        super().__init__()
        self._bank = FilterBank(n_octaves, bins_per_octave, sample_rate, int(secs_per_block * sample_rate), True)
        self.block_length = self._bank.block_length
        self.max_window_length = self._bank.max_window_length
        self.sample_rate = sample_rate
        self.hop_length = self.block_length / self.max_window_length
        self.n_bins = n_octaves * bins_per_octave
        # librosa.hz_to_midi written out (cqtwrapper.py:45)
        fmin = 12.0 * (math.log2((sample_rate / 2) / (2 ** n_octaves)) - math.log2(440.0)) + 69.0
        self.midi_freqs = fmin + np.arange(self.n_bins) / (bins_per_octave / 12)
        self._plans = {}

    # ---- plumbing ---------------------------------------------------------------------
    def _plan(self, device):
        key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
        if key not in self._plans:
            self._plans[key] = _Plan(self._bank, device, self.BLOCKS_PER_LAUNCH, self.LANES)
        return self._plans[key]

    # the buffers cqt_pytorch.CQT registers, as reference checkpoints carry them under `sliCQ.`
    CHECKPOINT_BUFFERS = ('windows', 'windows_range_indices', 'windows_inverse')

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        # A checkpoint of the reference carries cqt_pytorch's tables.  When all three are present the kernels are driven by
        # THEM (the transform the weights were trained with); otherwise the tables built from the constructor arguments stay.
        # Either way the entries are consumed here: this module has no parameters or buffers of its own.
        found = {name: state_dict[prefix + name] for name in self.CHECKPOINT_BUFFERS if prefix + name in state_dict}
        for key in [k for k in state_dict if k.startswith(prefix)]:
            state_dict.pop(key)
        if len(found) == len(self.CHECKPOINT_BUFFERS):
            w = found['windows']
            if tuple(w.shape) != (self.n_bins, self.max_window_length):
                raise ValueError(f'checkpoint {prefix}windows {tuple(w.shape)} does not fit this CQT '
                                 f'({self.n_bins} bins, max_window_length {self.max_window_length})')
            if bool(torch.count_nonzero(w)):        # all-zero placeholders: keep the constructed tables
                self.set_filter_bank(FilterBank.from_buffers(self.block_length, w.detach().cpu().numpy(),
                                                             found['windows_range_indices'].detach().cpu().numpy(),
                                                             found['windows_inverse'].detach().cpu().numpy()))
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    def set_filter_bank(self, bank):
        """Drive the kernels with other tables (same geometry): drops the device plans, which are rebuilt on next use."""
        if (bank.n_bins, bank.block_length, bank.max_window_length) != (self.n_bins, self.block_length, self.max_window_length):
            raise ValueError('filter bank geometry differs from this CQT')
        self._bank = bank
        self._plans = {}

    def __getstate__(self):
        # plans hold raw device handles (ctypes pointers cannot be pickled, and a copied handle would be freed twice):
        # torch.save(model) / copy.deepcopy(model), which the reference's training loop relies on (experiments/train.py:511),
        # carry the host tables only; plans are rebuilt lazily on the first call on a device.
        state = self.__dict__.copy()
        state['_plans'] = {}
        return state

    def _interleaved(self, coefficients):
        """(B, 2, F, T) real in any layout -> the (B, F, T, 2) contiguous buffer behind it (copy only if needed)."""
        c = coefficients.permute(0, 2, 3, 1)
        if c.dtype != torch.float32:
            c = c.float()
        return c if c.is_contiguous() else c.contiguous()

    # ---- transforms ---------------------------------------------------------------------
    def encode_interleaved(self, audio):
        """(B, 1, n*L) -> (B, F, n*M, 2) fp32 interleaved (re, im)."""
        _lib.require_cuda(audio, 'audio')
        if audio.dim() != 3 or audio.size(1) != 1:
            raise ValueError(f'audio must be (B, 1, T), got {tuple(audio.shape)}')
        if audio.size(-1) % self.block_length:
            raise ValueError(f'audio length {audio.size(-1)} is not a multiple of block_length {self.block_length} '
                             '(pad_to_block_length first)')
        audio = audio.detach().to(torch.float32).contiguous()
        B, n = audio.size(0), audio.size(-1) // self.block_length
        out = torch.empty((B, self.n_bins, n * self.max_window_length, 2), dtype=torch.float32, device=audio.device)
        if B * n:
            _lib.launch('tt_cqt_forward', self._plan(audio.device).handle, audio, B, n, out)
        return out

    def encode(self, audio):
        """cqt_pytorch.CQT.encode as used at cqtwrapper.py:67: complex (B, 1, F, T)."""
        with torch.no_grad():
            return torch.view_as_complex(self.encode_interleaved(audio)).unsqueeze(-3)

    def forward(self, audio):
        """CQT.forward (cqtwrapper.py:50-72): (B, 1, T) -> (B, 2, F, T') real/imaginary."""
        with torch.no_grad():
            return self.encode_interleaved(audio).permute(0, 3, 1, 2)

    def decode_raw(self, coefficients, normalise=False):
        """Synthesis; returns (audio (B,1,T), peak 0-dim device tensor = max|audio| before any normalisation)."""
        with torch.no_grad():
            if coefficients.is_complex():
                c = torch.view_as_real(coefficients.squeeze(-3).contiguous())
                if c.dtype != torch.float32:
                    c = c.float()
            else:
                c = self._interleaved(coefficients)
            _lib.require_cuda(c, 'coefficients')
            B, F, T, _ = c.shape
            if F != self.n_bins or T % self.max_window_length:
                raise ValueError(f'coefficients must be (B, 2, {self.n_bins}, k*{self.max_window_length})')
            n = T // self.max_window_length
            audio = torch.empty((B, 1, n * self.block_length), dtype=torch.float32, device=c.device)
            peak = torch.zeros((), dtype=torch.float32, device=c.device)
            if B * n:
                _lib.launch('tt_cqt_inverse', self._plan(c.device).handle, c, B, n, audio, peak, int(normalise))
        return audio, peak

    def decode(self, coefficients):
        """CQT.decode (cqtwrapper.py:184-213): synthesis + global infinity-norm normalise (no host sync here)."""
        return self.decode_raw(coefficients, normalise=True)[0]

    # ---- layout / element-wise helpers ----------------------------------------------------
    @staticmethod
    def to_real(coefficients):
        """cqtwrapper.py:74-97 (a view)."""
        return torch.view_as_real(coefficients.squeeze(-3)).transpose(-1, -2).transpose(-2, -3)

    @staticmethod
    def to_complex(coefficients):
        """cqtwrapper.py:99-120."""
        return torch.view_as_complex(coefficients.transpose(-3, -2).transpose(-2, -1).contiguous())

    @staticmethod
    def _magnitude(coefficients, apply_tanh):
        _lib.require_cuda(coefficients, 'coefficients')
        c = coefficients.detach().permute(0, 2, 3, 1)
        c = (c if c.dtype == torch.float32 else c.float())
        c = c if c.is_contiguous() else c.contiguous()
        out = torch.empty(c.shape[:-1], dtype=torch.float32, device=c.device)
        if out.numel():
            _lib.launch('tt_magnitude', c, out.numel(), int(apply_tanh), out)
        return out

    @staticmethod
    def to_magnitude(coefficients):
        """cqtwrapper.py:122-141: (B, 2, F, T) -> (B, F, T)."""
        return CQT._magnitude(coefficients, False)

    @staticmethod
    def to_decibels(magnitude, rescale=True):
        """cqtwrapper.py:143-182: per item, AmplitudeToDB(top_db=80), optional 0 dB ceiling and [0,1] rescale."""
        _lib.require_cuda(magnitude, 'magnitude')
        m = magnitude.detach().to(torch.float32).contiguous()
        out = torch.empty_like(m)
        B = m.size(0)
        if m.numel():
            scratch = torch.empty(B, dtype=torch.float32, device=m.device)
            _lib.launch('tt_to_decibels', m, B, m.numel() // B, int(rescale), out, scratch)
        return out

    # ---- host-side frame-grid helpers -----------------------------------------------------
    def pad_to_block_length(self, audio):
        """cqtwrapper.py:215-233."""
        return torch.nn.functional.pad(audio, (0, -audio.size(-1) % self.block_length))

    def get_expected_samples(self, t):
        """cqtwrapper.py:235-253."""
        return int(max(0, t) * self.sample_rate)

    def get_expected_frames(self, num_samples):
        """cqtwrapper.py:255-273."""
        return math.ceil((num_samples / self.block_length) * self.max_window_length)

    def get_times(self, n_frames):
        """cqtwrapper.py:275-293."""
        return np.arange(n_frames) * self.hop_length / self.sample_rate

    def get_midi_freqs(self):
        """cqtwrapper.py:295-308."""
        return self.midi_freqs
