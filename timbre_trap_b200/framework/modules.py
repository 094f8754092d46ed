"""
Drop-in for the autoencoder of `timbre_trap.framework.modules` (reference:
timbre_trap/framework/modules.py:23-777): `TimbreTrap`, `Encoder`, `Decoder`, `EncoderBlock`,
`DecoderBlock`, `ResidualConv2dBlock` with the reference's constructor signatures, attribute
names and state_dict keys (SURVEY.md A.4) - so reference checkpoints load unchanged - but every
convolution runs in the sm_100a kernels of csrc/conv_kernels.cu (bf16 operands, fp32 accumulate).

The torch.nn.Conv2d / ConvTranspose2d objects inside the blocks are PARAMETER HOLDERS only (same
names, shapes and default initialisation as the reference); their forward is never called.
Activations between layers live in the C8 planar bf16 layout (B, ceil(C/8), H, T, 8).
"""

import ctypes

import numpy as np
import torch
import torch.nn as nn

from .. import _lib
from . import ops
from . import packing as P
from .cqt import CQT
from .layer_grads import (_ActivationsFn, _Channel0ActivationsFn, _DownFn, _FiLMConvInFn, _HeadFn, _IndicatorFn, _InFn, _LatFn, _OutFn, _ResFn,
                          _SkipAddFn, _UpFn)
from .packing import _PackedCache       # also the name under which pickled modules refer to it

__all__ = ['TimbreTrap', 'TimbreTrapFiLM', 'FiLM', 'TimbreTrapMag', 'TimbreTrapMagDB', 'Encoder', 'Decoder', 'EncoderBlock', 'DecoderBlock',
           'ResidualConv2dBlock', 'shard_block_range', 'shard_audio']


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _n16(c):
    return max(16, P.pad8(c))


class ResidualConv2dBlock(nn.Module):
    """modules.py:721-777: y = x + ELU(conv1x1(ELU(conv3x3_dilated(x)))), one fused kernel."""

    def __init__(self, in_channels, out_channels, kernel_size=3, dilation=1):
        super().__init__()
        if in_channels != out_channels or kernel_size != 3:
            raise ValueError('timbre_trap_b200 implements the residual block as the reference uses it: C -> C, 3x3')
        self.conv1 = nn.Sequential(nn.Conv2d(in_channels, out_channels, kernel_size=kernel_size, padding='same', dilation=dilation),
                                   nn.ELU(inplace=True))
        self.conv2 = nn.Sequential(nn.Conv2d(out_channels, out_channels, kernel_size=1), nn.ELU(inplace=True))
        self.dilation = dilation
        self.channels = in_channels
        self.packed4 = False        # set by Encoder / Decoder for the first / last stage: (B, H, T, 4) activations
        self._caches = {}

    def _packed(self, mode):
        """mode: 'fold4' / 'fold2' / 'pairs' / 'planar' (csrc/res_rs.cu layouts 4 / 2 / 1 / 0)."""
        c1, c2 = self.conv1[0], self.conv2[0]
        args = (c1.weight, c1.bias, c2.weight, c2.bias)
        build = {'fold4': lambda: P.pack_res_rs_fold(*args, self.dilation, 4),
                 'fold2': lambda: P.pack_res_rs_fold(*args, self.dilation, 2),
                 'pairs': lambda: P.pack_res_rs_pairs(*args, self.dilation),
                 'planar': lambda: P.pack_res_rs(*args)}[mode]
        return self._caches.setdefault(mode, _PackedCache()).get(args, build)

    def forward_c8(self, x, out=None, mid_out=None, grad=False):
        """`grad`: through _ResFn (framework/layer_grads.py), whose forward is this call with `mid_out`; `out` is inference only."""
        if grad:
            if out is not None:
                raise ValueError('out= is for inference only')
            c1, c2 = self.conv1[0], self.conv2[0]
            return _ResFn.apply(x, c1.weight, c1.bias, c2.weight, c2.bias, lambda t, mid: self.forward_c8(t, mid_out=mid), self.channels,
                                self.dilation)
        # rows of C <= 8 tensors are folded to 16 values (4 or 2 frames per GEMM row) when T allows
        T = x.size(-2)
        if self.packed4:
            mode = 'fold4' if T % 4 == 0 else 'pairs'
        else:
            mode = 'fold2' if (self.channels <= 8 and T % 2 == 0) else 'planar'
        w1, w2, bias = self._packed(mode)
        return ops.res_block_rs(x, w1, w2, bias, self.channels, self.dilation, out=out, fold=mode.startswith('fold'), mid_out=mid_out)

    def forward(self, x):
        """(B, C, H, W) -> (B, C, H, W) fp32 (API parity; the fast paths stay in the internal layouts)."""
        if self.packed4:
            return P.from_p4(self.forward_c8(P.to_p4(x)), self.channels)
        return P.from_c8(self.forward_c8(P.to_c8(x)), self.channels)


class EncoderBlock(nn.Module):
    """modules.py:597-655: residual blocks with dilation 1, 2, 3, then a (4,1)/(2,1) strided conv + ELU."""

    def __init__(self, in_channels, out_channels, stride=2):
        super().__init__()
        if stride != 2:
            raise ValueError('stride 2 only (the reference never uses another value)')
        self.block1 = ResidualConv2dBlock(in_channels, in_channels, kernel_size=3, dilation=1)
        self.block2 = ResidualConv2dBlock(in_channels, in_channels, kernel_size=3, dilation=2)
        self.block3 = ResidualConv2dBlock(in_channels, in_channels, kernel_size=3, dilation=3)
        self.hop = stride
        self.win = 2 * stride
        self.sconv = nn.Sequential(nn.Conv2d(in_channels, out_channels, kernel_size=(self.win, 1), stride=(self.hop, 1)),
                                   nn.ELU(inplace=True))
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.packed4 = False
        self._cache = _PackedCache()

    def set_packed4(self, flag):
        """Input activations (and the three residual blocks) in the packed 4-channel layout; the output stays C8 planar."""
        self.packed4 = flag
        for blk in (self.block1, self.block2, self.block3):
            blk.packed4 = flag

    def forward_c8(self, x, grad=False):
        """`grad`: every layer through its autograd Function, and no buffer reused (the Functions keep their tensors for the backward)."""
        a = self.block1.forward_c8(x, grad=grad)
        b = self.block2.forward_c8(a, grad=grad)
        a = self.block3.forward_c8(b, out=None if grad else a, grad=grad)
        c = self.sconv[0]
        pack = P.pack_down_pairs if self.packed4 else P.pack_down_strip

        def run(t):
            (w,) = self._cache.get((c.weight, c.bias), lambda: (pack(c.weight, c.bias),))
            return ops.conv_down_strip(t, w, P.pad8(self.out_channels))
        return _DownFn.apply(a, c.weight, c.bias, run, self.in_channels, self.out_channels) if grad else run(a)

    def forward(self, x):
        return P.from_c8(self.forward_c8(P.to_p4(x) if self.packed4 else P.to_c8(x)), self.out_channels)


class DecoderBlock(nn.Module):
    """modules.py:658-718: (4,1)/(2,1) transposed conv (+output_padding) + ELU, then dilations 1, 2, 3."""

    def __init__(self, in_channels, out_channels, stride=2, padding=0):
        super().__init__()
        if stride != 2:
            raise ValueError('stride 2 only (the reference never uses another value)')
        self.hop = stride
        self.win = 2 * stride
        self.tconv = nn.Sequential(nn.ConvTranspose2d(in_channels, out_channels, kernel_size=(self.win, 1), stride=(self.hop, 1),
                                                      output_padding=(padding, 0)),
                                   nn.ELU(inplace=True))
        self.block1 = ResidualConv2dBlock(out_channels, out_channels, kernel_size=3, dilation=1)
        self.block2 = ResidualConv2dBlock(out_channels, out_channels, kernel_size=3, dilation=2)
        self.block3 = ResidualConv2dBlock(out_channels, out_channels, kernel_size=3, dilation=3)
        self.out_channels = out_channels
        self.out_pad = padding
        self.packed4 = False
        self._cache = _PackedCache()

    def set_packed4(self, flag):
        """Output activations (and the three residual blocks) in the packed 4-channel layout; the input stays C8 planar."""
        self.packed4 = flag
        for blk in (self.block1, self.block2, self.block3):
            blk.packed4 = flag

    def forward_c8(self, x, out=None, grad=False):
        """`out`: where the stage's result goes (e.g. a slice of the all-chunks buffer the fused convout / cross-fade reads), inference
        only.  `grad`: every layer through its autograd Function, and no buffer reused."""
        if grad and out is not None:
            raise ValueError('out= is for inference only')
        c = self.tconv[0]

        def run(t):
            (w,) = self._cache.get((c.weight, c.bias), lambda: (P.pack_up_strip(c.weight, c.bias),))
            return ops.conv_up_strip(t, w, P.pad8(self.out_channels), self.out_pad, packed4_out=self.packed4)
        a = _UpFn.apply(x, c.weight, c.bias, run, c.in_channels, c.out_channels) if grad else run(x)
        b = self.block1.forward_c8(a, grad=grad)
        a = self.block2.forward_c8(b, out=None if grad else a, grad=grad)
        return self.block3.forward_c8(a, out=None if grad else (b if out is None else out), grad=grad)

    def forward(self, x):
        y = self.forward_c8(P.to_c8(x))
        return P.from_p4(y, self.out_channels) if self.packed4 else P.from_c8(y, self.out_channels)


def _channels(model_complexity):
    return tuple(round(c * 2 ** (model_complexity - 1)) for c in (2, 4, 8, 16, 32))


def _check_channel_plan(channels):
    """The residual-block kernels exist for 8 / 16 / 32 padded channels (csrc/res_rs.cu): model_complexity 1 and 2 (the reference's
    base model, experiments/train.py:98).  Anything wider is rejected here, at construction, not at the first forward."""
    widest_res = max(channels[:4])
    if channels[0] > 8 or widest_res > 32 or max(channels) % 16:
        raise ValueError(f'timbre_trap_b200 supports model_complexity 1 and 2 (residual stages of at most 32 channels); the channel '
                         f'plan {tuple(channels)} has a {widest_res}-channel residual stage')


class Encoder(nn.Module):
    """modules.py:396-483."""

    def __init__(self, feature_size, latent_size=None, model_complexity=1):
        super().__init__()
        channels = _channels(model_complexity)
        if latent_size is None:
            latent_size = 32 * 2 ** (model_complexity - 1)
        _check_channel_plan(channels)
        self.convin = nn.Sequential(nn.Conv2d(2, channels[0], kernel_size=3, padding='same'), nn.ELU(inplace=True))
        self.block1 = EncoderBlock(channels[0], channels[1], stride=2)
        self.block2 = EncoderBlock(channels[1], channels[2], stride=2)
        self.block3 = EncoderBlock(channels[2], channels[3], stride=2)
        self.block4 = EncoderBlock(channels[3], channels[4], stride=2)
        embedding_size = feature_size
        for _ in range(4):
            embedding_size = embedding_size // 2 - 1
        self.convlat = nn.Conv2d(channels[4], latent_size, kernel_size=(embedding_size, 1))
        self.channels = channels
        self.latent_size = latent_size
        self.latent_pad = _latent_pad(latent_size)
        # first stage in the packed 4-channel layout (8 B per frame instead of the 16 B of channel-padded C8 planar)
        self.packed4 = channels[0] <= 4 and channels[1] <= 8
        self.block1.set_packed4(self.packed4)
        self._cache = _PackedCache()

    def _packed(self):
        ci, cl = self.convin[0], self.convlat

        def build():
            w = ci.weight.detach().float()
            if w.size(1) == 1:          # TimbreTrapMag / MagDB (modules.py:908-911): one input channel = pairs (x, 0) against (w, 0)
                w = torch.cat((w, torch.zeros_like(w)), dim=1)
            return w.contiguous(), ci.bias.detach().float().contiguous(), P.pack_lat(cl.weight, self.latent_pad), P.pad_vec(cl.bias, self.latent_pad)
        return self._cache.get((ci.weight, ci.bias, cl.weight, cl.bias), build)

    def forward_c8(self, coeffs_bft2, grad=False):
        """coeffs (B, F, T, 2) fp32 interleaved -> (latents C8 (B, Dp/8, 1, T, 8), [5 embeddings C8]).  `grad`: every layer through
        its autograd Function."""
        w_in, b_in, w_lat, b_lat = self._packed()
        ci, cl, ch = self.convin[0], self.convlat, self.channels

        def run_in(t):
            return ops.conv_in(t, w_in, b_in, ch[0], packed4=self.packed4)

        def run_lat(t):
            return ops.conv_lat(t, w_lat, b_lat, self.latent_pad)
        emb = [_InFn.apply(coeffs_bft2, ci.weight, ci.bias, run_in, ch[0]) if grad else run_in(coeffs_bft2)]
        for blk in (self.block1, self.block2, self.block3, self.block4):
            emb.append(blk.forward_c8(emb[-1], grad=grad))
        if grad:
            return _LatFn.apply(emb[-1], cl.weight, cl.bias, run_lat, ch[4], self.latent_size, self.latent_pad), emb
        return run_lat(emb[-1]), emb

    def forward(self, coefficients):
        """Encoder.forward (modules.py:448-483): (B, 2, F, T) -> (latents (B, D, T), embeddings, {}); (B, 1, F, T) for the
        magnitude variants, whose convin has one input channel."""
        _lib.require_cuda(coefficients, 'coefficients')
        if coefficients.size(1) != self.convin[0].in_channels:
            raise ValueError(f'expected {self.convin[0].in_channels} input channels, got {coefficients.size(1)}')
        with torch.no_grad():
            lat, emb = self.forward_c8(_interleave(coefficients))
            latents = P.from_c8(lat, self.latent_size).squeeze(-2)
            embeddings = [P.from_p4(e, c) if e.dim() == 4 else P.from_c8(e, c) for e, c in zip(emb, self.channels)]
        return latents, embeddings, dict()


class Decoder(nn.Module):
    """modules.py:486-594."""

    def __init__(self, feature_size, latent_size=None, model_complexity=1):
        super().__init__()
        channels = _channels(model_complexity)[::-1]
        _check_channel_plan(channels[::-1])
        if latent_size is None:
            latent_size = 32 * 2 ** (model_complexity - 1)
        padding = []
        embedding_size = feature_size
        for _ in range(4):
            padding.append(embedding_size % 2)
            embedding_size = embedding_size // 2 - 1
        padding.reverse()
        self.convin = nn.Sequential(nn.ConvTranspose2d(latent_size + 1, channels[0], kernel_size=(embedding_size, 1)), nn.ELU(inplace=True))
        self.block1 = DecoderBlock(channels[0], channels[1], stride=2, padding=padding[0])
        self.block2 = DecoderBlock(channels[1], channels[2], stride=2, padding=padding[1])
        self.block3 = DecoderBlock(channels[2], channels[3], stride=2, padding=padding[2])
        self.block4 = DecoderBlock(channels[3], channels[4], stride=2, padding=padding[3])
        self.convout = nn.Conv2d(channels[4], 2, kernel_size=3, padding='same')
        self.channels = channels
        self.latent_size = latent_size
        self.latent_pad = _latent_pad(latent_size)
        self.embedding_size = embedding_size
        self.packed4 = channels[4] <= 4 and channels[3] <= 8
        self.block4.set_packed4(self.packed4)
        self._cache = _PackedCache()
        self._film = None           # set by TimbreTrapFiLM: the FiLM layer folded into convin's packed weights

    def _embeddings_internal(self, encoder_embeddings):
        """(B, C, H, T) encoder embeddings (API form) -> the internal layouts the decoder stages use."""
        out = [P.to_c8(e) for e in encoder_embeddings]
        if self.packed4:
            out[0] = P.to_p4(encoder_embeddings[0])
        return out

    def _packed(self):
        """((w_in[transcribe], w_in[reconstruct]), (bias table[transcribe], [reconstruct]), w_out, b_out)."""
        ci, co = self.convin[0], self.convout
        film = self._film
        params = (ci.weight, ci.bias, co.weight, co.bias)
        if film is not None:
            params += (film.gamma.weight, film.gamma.bias, film.beta.weight, film.beta.bias)

        def build():
            if film is None:
                w, tables = P.pack_deconv_in(ci.weight, ci.bias, self.latent_pad)
                ws, tables = (w, w), (tables[0], tables[1])
            else:
                ws, tables = [], []
                for transcribe in (True, False):
                    # TimbreTrapFiLM.decode (modules.py:835-838): condition = one-hot [transcribe, not transcribe]
                    cond = torch.tensor([float(transcribe), float(not transcribe)], dtype=film.gamma.weight.dtype, device=ci.weight.device)
                    w, t = P.pack_deconv_in_film(ci.weight, ci.bias, film.gamma(cond), film.beta(cond), self.latent_pad)
                    ws.append(w)
                    tables.append(t)
            w_out, b_out = co.weight.detach().float(), co.bias.detach().float()
            if w_out.size(0) == 1:      # TimbreTrapMag / MagDB (modules.py:913): one output channel = channel 0 of the pair
                w_out, b_out = torch.cat((w_out, torch.zeros_like(w_out)), dim=0), torch.cat((b_out, torch.zeros_like(b_out)))
            return tuple(ws), tuple(tables), w_out.contiguous(), b_out.contiguous()
        return self._cache.get(params, build)

    def last_stage_c8(self, lat_c8, reconstruct, skips=None, out=None, convin=None, grad=False):
        """Everything before `convout`: latents C8 (B, Dp/8, 1, T, 8) (without the indicator channel) -> the last stage's
        activations in their internal layout (packed4 (B, F, T, 4) for the supported channel plans), written to `out` if given.
        `grad`: every layer through its autograd Function, and no buffer reused; `out` and `convin` are inference only."""
        if grad and (out is not None or convin is not None):
            raise ValueError('out= and convin= are for inference only')
        w_in, tables, _, _ = self._packed()
        sw = 1 if reconstruct else 0
        w_sel, t_sel = (w_in[sw], tables[sw]) if convin is None else convin
        ci, film = self.convin[0], self._film

        def run_in(t):
            return ops.deconv_in(t, w_sel, t_sel, P.pad8(self.channels[0]), self.embedding_size)
        if not grad:
            x = run_in(lat_c8)
        elif film is None:
            x = _IndicatorFn.apply(lat_c8, ci.weight, ci.bias, run_in, 1.0 if reconstruct else 0.0, self.latent_size, self.channels[0])
        else:
            # TimbreTrapFiLM.decode (modules.py:835-838): condition = one-hot [transcribe, not transcribe]
            x = _FiLMConvInFn.apply(lat_c8, ci.weight, ci.bias, film.gamma.weight, film.gamma.bias, film.beta.weight, film.beta.bias, run_in,
                                    1 if reconstruct else 0, self.latent_size, self.channels[0])
        blocks = (self.block1, self.block2, self.block3, self.block4)
        for i, blk in enumerate(blocks):
            if skips is not None:                      # modules.py:568-585: x + weight * encoder embedding, one native pass (in place)
                w, e = skips[-1 - i]
                x = _SkipAddFn.apply(x, e, w) if grad else ops.add_scaled(x, e, w, out=x)
            last = i == len(blocks) - 1
            x = blk.forward_c8(x, out=out if (last and skips is None) else None, grad=grad)
        if skips is not None:
            w, e = skips[0]
            x = _SkipAddFn.apply(x, e, w) if grad else ops.add_scaled(x, e, w, out=out if out is not None else x)
        return x

    def forward_c8(self, lat_c8, reconstruct, skips=None, convin=None, grad=False):
        """latents C8 (B, Dp/8, 1, T, 8) (without the indicator channel) -> coefficients (B, F, T, 2) fp32 interleaved.  `grad`: every
        layer through its autograd Function; `convin` is inference only."""
        _, _, w_out, b_out = self._packed()
        x = self.last_stage_c8(lat_c8, reconstruct, skips, convin=convin, grad=grad)
        co, c = self.convout, self.channels[4]

        def run_out(t):
            return ops.conv_out(t, w_out, b_out, c)
        return _OutFn.apply(x, co.weight, co.bias, run_out, c) if grad else run_out(x)

    def forward(self, latents, encoder_embeddings=None):
        """Decoder.forward (modules.py:545-594): latents (B, D+1, T) WITH the indicator channel -> (B, 2, F, T)."""
        _lib.require_cuda(latents, 'latents')
        if self._film is not None:
            # TimbreTrapFiLM: the decoder proper takes latents the FiLM layer has ALREADY been applied to and has no indicator channel
            # (modules.py:838-840); model.decode() folds the layer into convin instead
            with torch.no_grad():
                ci = self.convin[0]
                d = ci.weight.size(0)
                plain = P.pack_deconv_in_film(ci.weight, ci.bias, torch.ones(d, device=latents.device), torch.zeros(d, device=latents.device),
                                              self.latent_pad)
                skips = None if encoder_embeddings is None else _unit_skips(self._embeddings_internal(encoder_embeddings))
                pairs = self.forward_c8(_latents_to_c8(latents, self.latent_pad), True, skips, convin=plain)
            return pairs.permute(0, 3, 1, 2)
        with torch.no_grad():
            flag = latents[:, -1]
            is_one, is_zero = bool((flag == 1).all()), bool((flag == 0).all())
            if not (is_one or is_zero):
                raise ValueError('the indicator channel must be all ones (reconstruct) or all zeros (transcribe), as '
                                 'TimbreTrap.decode builds it (modules.py:139-142)')
            lat = _latents_to_c8(latents[:, :-1], self.latent_pad)
            skips = None if encoder_embeddings is None else _unit_skips(self._embeddings_internal(encoder_embeddings))
            pairs = self.forward_c8(lat, is_one, skips)
            return pairs.permute(0, 3, 1, 2) if self.convout.out_channels == 2 else pairs[..., :1].permute(0, 3, 1, 2)


def _interleave(coefficients):
    """(B, 2, F, T) real (any strides) -> contiguous (B, F, T, 2) fp32 (free for the CQT's own output); a one-channel feature map
    (B, 1, F, T) becomes pairs (x, 0)."""
    if coefficients.size(1) == 1:
        return ops.widen(coefficients[:, 0])
    c = coefficients.detach().permute(0, 2, 3, 1)
    if c.dtype != torch.float32:
        c = c.float()
    return c if c.is_contiguous() else c.contiguous()


def _no_autocast():
    """The model's own code runs outside autocast: the ATen pieces that build the packed weights (FiLM's nn.Linear, the skip-weight
    products, re-layouts) would otherwise store autocast-dependent values in caches whose keys do not record the autocast state."""
    return torch.autocast('cuda', enabled=False)


def _unit_skips(embeddings_internal):
    """Already-weighted embeddings (the API form of Decoder.forward / TimbreTrap.decode) as (weight 1, embedding) pairs."""
    one = torch.ones((), dtype=torch.float32, device=embeddings_internal[0].device)
    return [(one, e) for e in embeddings_internal]


def _latent_pad(latent_size):
    """Latent channels as the (H, 1)-kernel layers see them: zero-padded to the next GEMM width the kernels are built for."""
    for n in (16, 32, 64, 128, 256):
        if latent_size <= n:
            return n
    raise ValueError(f'latent_size {latent_size} is not supported (at most 256)')


def _latents_to_c8(latents, latent_pad, grad=False):
    """(B, D, T) -> C8 planar (B, Dp/8, 1, T, 8) bf16.  `grad`: the re-layout stays on the autograd graph of `latents`."""
    B, D, T = latents.shape
    x = latents.float() if grad else latents.detach().float()
    if D != latent_pad:
        x = torch.nn.functional.pad(x, (0, 0, 0, latent_pad - D))
    return x.reshape(B, latent_pad // 8, 8, 1, T).permute(0, 1, 3, 4, 2).contiguous().to(torch.bfloat16)


def shard_block_range(n_blocks, rank, world):
    """Contiguous, balanced ranges of blocks: rank r owns [r * n // world, (r + 1) * n // world)."""
    return rank * n_blocks // world, (rank + 1) * n_blocks // world


def shard_audio(padded, block_length, rank, world):
    """padded (B, 1, n * L): the samples rank `rank` needs for its output blocks [b0, b1) - those blocks plus half a block on
    either side (zeros beyond the ends of the clip, exactly the padding of the unsharded loop, modules.py:226-234)."""
    L, hop = block_length, block_length // 2
    b0, b1 = shard_block_range(padded.size(-1) // L, rank, world)
    haloed = torch.nn.functional.pad(padded, [hop, hop])
    return haloed[..., b0 * L: b1 * L + 2 * hop], b0, b1


def _resolve_group(group, rank=None, world=None):
    """(group, rank, world) of a sharded call.  With explicit `rank` / `world` and no group the caller emulates the ranks one after
    the other (no collective).  Otherwise the ranks are those of `group`, or of the DEFAULT process group when torch.distributed is
    initialised - so that `model.transcribe_sharded(audio)` under torchrun shards AND gathers over the same ranks."""
    if rank is not None and world is not None:
        return group, rank, world
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        if group is not None:
            raise ValueError('a process group was passed but torch.distributed is not initialised')
        return None, 0, 1
    if group is None:
        group = dist.group.WORLD
    return group, dist.get_rank(group), dist.get_world_size(group)


def _gather_frames(local, dim, per_block, audio, block_length, group, world):
    """all_gather of per-rank results whose extent along `dim` is (blocks of the rank) * per_block (ranks may differ by one block)."""
    if group is None or world == 1:
        return local
    import torch.distributed as dist
    n_blocks = -(-audio.size(-1) // block_length)
    counts = [shard_block_range(n_blocks, r, world) for r in range(world)]
    most = max(b1 - b0 for b0, b1 in counts) * per_block
    shape = list(local.shape)
    shape[dim] = most
    mine = torch.zeros(shape, dtype=local.dtype, device=local.device)
    mine.narrow(dim, 0, local.size(dim)).copy_(local)
    parts = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(parts, mine, group=group)
    return torch.cat([p.narrow(dim, 0, (b1 - b0) * per_block) for p, (b0, b1) in zip(parts, counts)], dim=dim)


class TimbreTrap(nn.Module):
    """modules.py:23-393.  Same public surface; `sliCQ` is the CQT module (every reference script uses that name)."""

    # chunks per kernel batch of the chunked paths (bounds activation memory: ~2.3 GB per live tensor at 256 chunks)
    MAX_CHUNKS_PER_BATCH = 256
    # convout + Hann cross-fade + trim (+ tanh|.|) as one kernel over all chunks; False = per-chunk convout, then tt_chunk_crossfade
    # (same arithmetic in the same order: results are bit-identical, tests/test_model_gpu.py)
    FUSE_CONVOUT_CROSSFADE = True

    def __init__(self, sample_rate, n_octaves, bins_per_octave, secs_per_block=3, latent_size=None, model_complexity=1,
                 skip_connections=False):
        nn.Module.__init__(self)
        self.sliCQ = CQT(n_octaves=n_octaves, bins_per_octave=bins_per_octave, sample_rate=sample_rate, secs_per_block=secs_per_block)
        self.encoder = Encoder(feature_size=self.sliCQ.n_bins, latent_size=latent_size, model_complexity=model_complexity)
        self.decoder = Decoder(feature_size=self.sliCQ.n_bins, latent_size=latent_size, model_complexity=model_complexity)
        self.skip_weights = torch.nn.Parameter(torch.ones(5)) if skip_connections else None
        self._windows = {}
        self._warned_local_peak = False

    def __getstate__(self):
        state = self.__dict__.copy()
        state['_windows'] = {}                     # per-device Hann windows are rebuilt on demand
        return state

    # ---- C8 fast paths -----------------------------------------------------------------------------
    def _skips_c8(self, emb):
        """apply_skip_connections (modules.py:95-117) for the internal layouts: (learnable weight, embedding) pairs - the product is
        formed inside the one-pass add kernel (tt_add_scaled_bf16)."""
        if self.skip_weights is None:
            return None
        return [(self.skip_weights[i], e) for i, e in enumerate(emb)]

    def _features(self, audio):
        """audio (B, 1, n*L) -> the encoder's input as interleaved (B, F, T, 2) fp32: the CQT coefficients (modules.py:88)."""
        return self.sliCQ.encode_interleaved(audio)

    # output head of the variant (tt_channel0_activation mode; None = the two-channel coefficients as they are), and the mode of its
    # to_activations on the head's output (None = tanh|.| of the two-channel coefficients)
    HEAD_MODE = None
    ACTIVATIONS_MODE = None

    def _graph(self):
        """Whether forward / encode / decode build an autograd graph: in train mode with grad mode on.  In eval mode or under no_grad
        they run the inference path (the same launches, buffer reuse and outputs, no graph)."""
        return self.training and torch.is_grad_enabled()

    def _head(self, pairs, grad=False):
        """decoder output (B, F, T, 2) interleaved -> what `decode` returns: (B, 2, F, T) view, or (B, 1, F, T) for the magnitude variants.
        `grad`: the head through its autograd Function."""
        if self.HEAD_MODE is None:
            return pairs.permute(0, 3, 1, 2)
        if grad:
            return _Channel0ActivationsFn.apply(pairs, self.HEAD_MODE).unsqueeze(1)
        return ops.channel0(pairs, self.HEAD_MODE).unsqueeze(1)

    def _codes(self, audio):
        """audio (B, 1, n*L) -> (latents C8, skips C8 or None)."""
        lat, emb = self.encoder.forward_c8(self._features(audio))
        return lat, self._skips_c8(emb)

    def _passes(self, features, grad=False):
        """Encode the encoder input (B, F, T, 2), decode for the reconstruction and for the transcription (modules.py:338-393) ->
        (reconstruction, transcription, latents C8); the decoder outputs are pairs (B, F, T, 2) after the variant's head, a one-channel
        output h as (h, 0).  The consistency pass is this method again on the transcription.  `grad`: every layer through its autograd
        Function (framework/layer_grads.py), as the loss step runs it."""
        lat, emb = self.encoder.forward_c8(features, grad=grad)
        skips = self._skips_c8(emb)
        outs = []
        for reconstruct in (True, False):
            y = self.decoder.forward_c8(lat, reconstruct, skips, grad=grad)
            if self.HEAD_MODE is not None:
                y = _HeadFn.apply(y, self.HEAD_MODE) if grad else ops.widen(ops.channel0(y, self.HEAD_MODE))
            outs.append(y)
        return outs[0], outs[1], lat

    def _output(self, pairs, grad=False):
        """A decoder output of _passes -> what `forward` returns: (B, 2, F, T) view, or (B, 1, F, T) for the magnitude variants.
        `grad`: channel 0 through its autograd Function."""
        if self.HEAD_MODE is None:
            return pairs.permute(0, 3, 1, 2)
        if grad:
            return _Channel0ActivationsFn.apply(pairs, 0).unsqueeze(1)
        return ops.channel0(pairs, 0).unsqueeze(1)          # mode 0: channel 0 as it is

    # ---- reference API -------------------------------------------------------------------------------
    def encode(self, audio):
        """modules.py:67-93: audio (B, 1, N) -> (latents (B, D, T), embeddings [(B, C, H, T)], {}).  In train mode with grad mode on the
        result carries an autograd graph to the encoder's parameters (none to the audio: the CQT has no backward, as in the reference);
        in eval mode or under no_grad it is inference."""
        _lib.require_cuda(audio, 'audio')
        grad = self._graph()
        with _no_autocast(), torch.set_grad_enabled(grad):
            lat, emb = self.encoder.forward_c8(self._features(audio), grad=grad)
            latents = P.from_c8(lat, self.encoder.latent_size).squeeze(-2)
            embeddings = [P.from_p4(e, c) if e.dim() == 4 else P.from_c8(e, c) for e, c in zip(emb, self.encoder.channels)]
        return latents, embeddings, dict()

    def apply_skip_connections(self, embeddings):
        """modules.py:95-117."""
        if self.skip_weights is not None:
            return [self.skip_weights[i] * e for i, e in enumerate(embeddings)]
        return None

    def decode(self, latents, embeddings=None, transcribe=False):
        """modules.py:119-147: latents (B, D, T) -> logits (B, 2, F, T) ((B, 1, F, T) for the magnitude variants).  In train mode with
        grad mode on the result carries an autograd graph to the decoder's parameters and to `latents` and `embeddings` where they
        require grad; in eval mode or under no_grad it is inference."""
        _lib.require_cuda(latents, 'latents')
        grad = self._graph()
        with _no_autocast(), torch.set_grad_enabled(grad):
            lat = _latents_to_c8(latents, self.decoder.latent_pad, grad=grad)
            skips = None if embeddings is None else _unit_skips(self.decoder._embeddings_internal(embeddings))
            return self._head(self.decoder.forward_c8(lat, not transcribe, skips, grad=grad), grad)

    def _inference(self, audio, transcribe=False):
        """modules.py:149-177."""
        with torch.no_grad():
            lat, skips = self._codes(audio)
            return self._head(self.decoder.forward_c8(lat, not transcribe, skips))

    def inference(self, audio, transcribe=False):
        """modules.py:179-202."""
        return self._inference(self.sliCQ.pad_to_block_length(audio), transcribe)

    def _window(self, device):
        key = (device.type, device.index)
        if key not in self._windows:
            self._windows[key] = torch.signal.windows.hann(self.sliCQ.max_window_length, device=device)
        return self._windows[key]

    def _chunks(self, audio, prepadded=False):
        """Pad and slice audio into 50 %-overlapped blocks (modules.py:226-234, 247-253): (B*n_chunks, 1, L), n_chunks.
        prepadded: `audio` already is a whole number of blocks plus the half-block on either side (a shard of a longer clip
        with its true neighbourhood, see shard_audio)."""
        L = self.sliCQ.block_length
        hop = L // 2
        if not prepadded:
            audio = self.sliCQ.pad_to_block_length(audio)
            audio = torch.nn.functional.pad(audio, [hop] * 2)
        elif (audio.size(-1) - 2 * hop) % L:
            raise ValueError(f'a pre-padded shard must hold n * {L} + {2 * hop} samples, got {audio.size(-1)}')
        n_chunks = (audio.size(-1) - hop) // hop
        chunks = audio.unfold(-1, L, hop)[:, :, :n_chunks]                 # (B, 1, n_chunks, L) view
        return chunks.reshape(audio.size(0) * n_chunks, 1, L), n_chunks

    def _fused_convout(self):
        """Whether the chunked paths run convout + cross-fade as one kernel (tt_conv_out_crossfade) on the packed last stage."""
        return self.FUSE_CONVOUT_CROSSFADE and self.decoder.packed4 and self.sliCQ.max_window_length % 8 == 0 and self.HEAD_MODE is None

    def _chunked(self, audio, want_transcription, want_reconstruction, activations=True, prepadded=False, on_activations=None):
        """
        Batched form of chunked_inference (modules.py:204-269) for one or both switch settings with a shared
        encoder pass.  Returns (transcription, reconstruction) coefficient tensors (B, F, T, 2) interleaved - or the
        activations (B, F, T) for the transcription when `activations` - None where not requested.

        The last decoder stage of every chunk goes into one (B * n_chunks, F, M, 4) bf16 buffer per output; `convout`, the Hann
        cross-fade, the trim and (for activations) tanh|.| then run as ONE kernel over it (tt_conv_out_crossfade): the
        per-chunk fp32 coefficients of the reference's loop never exist.

        `on_activations(lo, hi, activations[lo:hi])` (fused path only): called as soon as the clips [lo, hi) have all their chunks
        through the decoder - their activations are produced right then, while the remaining chunk batches still compute, so a
        caller that streams results off the device (framework.HostPipeline) can start copying early.
        """
        _lib.require_cuda(audio, 'audio')
        with torch.no_grad():
            B, F, M = audio.size(0), self.sliCQ.n_bins, self.sliCQ.max_window_length
            chunks, n_chunks = self._chunks(audio.detach().float(), prepadded)
            n_out = (n_chunks - 1) * (M // 2)
            window = self._window(audio.device)
            fused = self._fused_convout()
            wants = (want_transcription, want_reconstruction)
            if fused:
                stages = [torch.empty((B * n_chunks, F, M, 4), dtype=torch.bfloat16, device=audio.device) if w else None for w in wants]
            else:
                stages = [torch.empty((B * n_chunks, F, M, 2), dtype=torch.float32, device=audio.device) if w else None for w in wants]
            step = self.MAX_CHUNKS_PER_BATCH
            early = on_activations is not None and fused and want_transcription and activations
            if early:
                act_early = torch.empty((B, F, n_out), dtype=torch.float32, device=audio.device)
                emitted = 0
            for c0 in range(0, B * n_chunks, step):
                lat, skips = self._codes(chunks[c0:c0 + step])
                for stage, reconstruct in zip(stages, (False, True)):
                    if stage is None:
                        continue
                    if fused:
                        self.decoder.last_stage_c8(lat, reconstruct, skips, out=stage[c0:c0 + step])
                    else:
                        y = self.decoder.forward_c8(lat, reconstruct, skips)
                        if self.HEAD_MODE is not None:
                            # the reference's loop adds the variant's ONE output channel into its hard-coded two-channel buffer
                            # (modules.py:244, 259-263): broadcast, i.e. both channels carry the head's output
                            y = ops.channel0(y, self.HEAD_MODE).unsqueeze(-1).expand(-1, -1, -1, 2)
                        stage[c0:c0 + step] = y
                if early:
                    done = min(B, (c0 + step) // n_chunks)            # clips whose chunks have all been decoded
                    if done > emitted:
                        self._convout_crossfade(stages[0], emitted, done, n_chunks, window, None, act_early)
                        on_activations(emitted, done, act_early[emitted:done])
                        emitted = done
            _, _, w_out, b_out = self.decoder._packed()
            results = []
            for stage, want_act in zip(stages, (activations, False)):
                if stage is None:
                    results.append(None)
                    continue
                if early and want_act:
                    results.append(act_early)
                    continue
                as_act = want_act and self.HEAD_MODE is None         # the fused tanh|.| is the BASE model's to_activations
                if as_act:
                    res = torch.empty((B, F, n_out), dtype=torch.float32, device=audio.device)
                    args = (None, ctypes.c_void_p(res.data_ptr()))
                else:
                    res = torch.empty((B, F, n_out, 2), dtype=torch.float32, device=audio.device)
                    args = (ctypes.c_void_p(res.data_ptr()), None)
                stream = ctypes.c_void_p(torch.cuda.current_stream(audio.device).cuda_stream)
                with torch.cuda.device(audio.device):
                    if fused:
                        _lib.check(_lib.lib().tt_conv_out_crossfade(ctypes.c_void_p(stage.data_ptr()), ctypes.c_void_p(window.data_ptr()),
                                                                    ctypes.c_void_p(w_out.data_ptr()), ctypes.c_void_p(b_out.data_ptr()),
                                                                    B, n_chunks, self.decoder.channels[4], F, M, args[0], args[1], stream))
                    else:
                        _lib.check(_lib.lib().tt_chunk_crossfade(ctypes.c_void_p(stage.data_ptr()), ctypes.c_void_p(window.data_ptr()),
                                                                 B, n_chunks, F, M, args[0], args[1], stream))
                if want_act and not as_act:
                    res = self.to_activations(res.permute(0, 3, 1, 2))       # a variant's own activation function
                results.append(res)
            return results

    def _convout_crossfade(self, stage, lo, hi, n_chunks, window, out_coeffs, out_act):
        """tt_conv_out_crossfade over the clips [lo, hi) of a (B * n_chunks, F, M, 4) stage buffer."""
        F, M = self.sliCQ.n_bins, self.sliCQ.max_window_length
        _, _, w_out, b_out = self.decoder._packed()
        sub = stage[lo * n_chunks: hi * n_chunks]
        with torch.cuda.device(stage.device):
            _lib.check(_lib.lib().tt_conv_out_crossfade(ctypes.c_void_p(sub.data_ptr()), ctypes.c_void_p(window.data_ptr()),
                                                        ctypes.c_void_p(w_out.data_ptr()), ctypes.c_void_p(b_out.data_ptr()),
                                                        hi - lo, n_chunks, self.decoder.channels[4], F, M,
                                                        None if out_coeffs is None else ctypes.c_void_p(out_coeffs[lo:hi].data_ptr()),
                                                        None if out_act is None else ctypes.c_void_p(out_act[lo:hi].data_ptr()),
                                                        ctypes.c_void_p(torch.cuda.current_stream(stage.device).cuda_stream)))

    def chunked_inference(self, audio, transcribe=False):
        """modules.py:204-269: (B, 1, N) -> (B, 2, F, T) cross-faded coefficients."""
        trn, rec = self._chunked(audio, transcribe, not transcribe, activations=False)
        return (trn if transcribe else rec).permute(0, 3, 1, 2)

    def to_activations(self, coefficients):
        """modules.py:271-289: tanh|c| of (B, 2, F, T) coefficients -> (B, F, T).  Differentiable (tt_activations_bwd) when grad mode is on
        and the coefficients require grad: `forward`'s outputs are views of interleaved pairs and go in as they are, other tensors are
        copied into pairs first."""
        if torch.is_grad_enabled() and coefficients.requires_grad:
            _lib.require_cuda(coefficients, 'coefficients')
            pairs = coefficients.permute(0, 2, 3, 1)
            if pairs.dtype != torch.float32 or not pairs.is_contiguous():
                pairs = pairs.float().contiguous()
            return _ActivationsFn.apply(pairs)
        return CQT._magnitude(coefficients, True)

    def transcribe(self, audio):
        """modules.py:292-313: (B, 1, N) -> activations (B, F, T) in [0, 1)."""
        return self._chunked(audio, True, False)[0]

    def _decode_shared_peak(self, coefficients, group):
        """
        CQT.decode with the reference's GLOBAL infinity-norm normalise (cqtwrapper.py:209-211) when the batch is sharded
        over the ranks of `group`: one scalar MAX all-reduce of the per-rank peaks, then a local scale.
        """
        if group is None:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 and not self._warned_local_peak:
                # the caller shards the batch by hand but asks for a rank-local normalise: legal (independent clips), but say so once
                import warnings
                warnings.warn('reconstruct(group=None) under torch.distributed normalises by the LOCAL peak of this rank; pass '
                              'group=... for the reference\'s global peak (cqtwrapper.py:209-211) over a sharded batch')
                self._warned_local_peak = True
            return self.sliCQ.decode(coefficients)
        import torch.distributed as dist
        audio, peak = self.sliCQ.decode_raw(coefficients, normalise=False)
        dist.all_reduce(peak, op=dist.ReduceOp.MAX, group=group)
        with torch.cuda.device(audio.device):
            _lib.check(_lib.lib().tt_scale_by_peak(ctypes.c_void_p(audio.data_ptr()), audio.numel(), ctypes.c_void_p(peak.data_ptr()),
                                                   ctypes.c_void_p(torch.cuda.current_stream(audio.device).cuda_stream)))
        return audio

    def reconstruct(self, audio_in, group=None):
        """modules.py:315-336: (B, 1, N) -> audio (B, 1, N') in [-1, 1].  `group`: see _decode_shared_peak."""
        return self._decode_shared_peak(self._chunked(audio_in, False, True)[1].permute(0, 3, 1, 2), group)

    def transcribe_and_reconstruct(self, audio, group=None, on_activations=None):
        """Both outputs of transcribe() and reconstruct() from ONE encoder pass (not in the reference, which runs two).
        `on_activations`: see _chunked (early hand-over of finished clips' activations; the returned tensors are the same)."""
        act, rec = self._chunked(audio, True, True, on_activations=on_activations)
        return act, self._decode_shared_peak(rec.permute(0, 3, 1, 2), group)

    # ---- many clips of different lengths in one batched pass ----------------------------------------------------------------
    # The clips' chunks are cut straight from the clips by one kernel (tt_gather_chunks) and run through the encoder / decoder in
    # batches of MAX_CHUNKS_PER_BATCH that cross clip boundaries; the cross-fade, the inverse CQT and the normalise read a clip table
    # (int32 prefix sums of chunks and blocks per clip), so the launches follow the number of chunks, not of clips.  Clips go in
    # groups of whole clips of at most MAX_CHUNKS_PER_GROUP chunks (or the longest clip's, if more): the per-chunk stage buffers
    # (4.4 MB per chunk at the base model) stay bounded whatever the number of clips.
    MAX_CHUNKS_PER_GROUP = 1024

    def transcribe_many(self, clips):
        """transcribe() of each of a list of clips of any lengths in one batched pass: `clips` (N_i,) or (1, N_i) CUDA tensors on one
        device -> a list of activations, the i-th equal bit for bit to transcribe(clips[i].view(1, 1, -1))[0].  Views of one buffer."""
        return self._many(clips, True, False)[0]

    def reconstruct_many(self, clips):
        """reconstruct() of each clip (see transcribe_many) -> a list of (1, N_i') audio, each normalised by its OWN peak - what
        reconstruct(clips[i].view(1, 1, -1))[0] returns, bit for bit (a silent clip comes back as zeros).  Views of one buffer."""
        return self._many(clips, False, True)[1]

    def transcribe_and_reconstruct_many(self, clips):
        """Both lists of transcribe_many and reconstruct_many from ONE encoder pass."""
        return self._many(clips, True, True)

    def _clip_table(self, clips):
        """Validate a list of clips -> (flat fp32 contiguous clips, samples, blocks, chunks per clip as int64 numpy arrays)."""
        device, flat = None, []
        for i, c in enumerate(clips):
            _lib.require_cuda(c, f'clips[{i}]')
            if not (c.dim() == 1 or (c.dim() == 2 and c.size(0) == 1)):
                raise ValueError(f'clips[{i}]: expected a mono clip of shape (N,) or (1, N), got {tuple(c.shape)}')
            if c.numel() == 0:
                raise ValueError(f'clips[{i}] is empty')
            if device is None:
                device = c.device
            elif c.device != device:
                raise ValueError(f'clips[{i}] is on {c.device}, clips[0] on {device}: all clips must be on one device')
            x = c.detach().reshape(-1)
            flat.append((x if x.dtype == torch.float32 else x.float()).contiguous())
        L, hop = self.sliCQ.block_length, self.sliCQ.block_length // 2
        samples = np.array([x.numel() for x in flat], dtype=np.int64)
        blocks = -(-samples // L)
        chunks = (blocks * L + hop) // hop              # _chunks: (n L + 2 hop - hop) // hop per clip
        return flat, samples, blocks, chunks

    def _many(self, clips, want_transcription, want_reconstruction):
        """(activations list or None, audio list or None) of the *_many calls."""
        clips = list(clips)
        if not clips:
            return [] if want_transcription else None, [] if want_reconstruction else None
        flat, samples, blocks, chunks = self._clip_table(clips)
        device = flat[0].device
        n = len(flat)
        F, M, L = self.sliCQ.n_bins, self.sliCQ.max_window_length, self.sliCQ.block_length
        half = M // 2
        chunk0 = np.concatenate(([0], np.cumsum(chunks)))
        block0 = np.concatenate(([0], np.cumsum(blocks)))
        out0 = np.concatenate(([0], np.cumsum((chunks - 1) * half)))          # first output frame of each clip
        # groups of whole clips: [groups[g], groups[g + 1])
        cap = max(self.MAX_CHUNKS_PER_GROUP, int(chunks.max()))
        groups = [0]
        for i in range(n):
            if chunk0[i + 1] - chunk0[groups[-1]] > cap:
                groups.append(i)
        groups.append(n)
        rows = max(int(chunk0[groups[g + 1]] - chunk0[groups[g]]) for g in range(len(groups) - 1))
        with torch.no_grad(), torch.cuda.device(device):
            tab = torch.from_numpy(np.concatenate((chunk0, block0)).astype(np.int32)).to(device)
            clip_tab = torch.from_numpy(np.stack((np.array([x.data_ptr() for x in flat], dtype=np.int64), samples), 1)).to(device)
            t_chunk0, t_block0 = tab[:n + 1], tab[n + 1:]
            stream = ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)
            window = self._window(device)
            fused = self._fused_convout()
            as_act = self.HEAD_MODE is None                  # the BASE model's tanh|.| is fused into the cross-fade
            _, _, w_out, b_out = self.decoder._packed()
            step = self.MAX_CHUNKS_PER_BATCH
            f32 = dict(dtype=torch.float32, device=device)
            batch = torch.empty((min(step, rows), L), **f32)
            wants = (want_transcription, want_reconstruction)
            if fused:
                stages = [torch.empty((rows, F, M, 4), dtype=torch.bfloat16, device=device) if w else None for w in wants]
            else:
                stages = [torch.empty((rows, F, M, 2), **f32) if w else None for w in wants]
            total_out = int(out0[-1])
            trn = torch.empty((F * total_out * (1 if as_act else 2),), **f32) if want_transcription else None
            audio = torch.empty((int(block0[-1]) * L,), **f32) if want_reconstruction else None
            peaks = torch.empty((n,), **f32) if want_reconstruction else None
            for g in range(len(groups) - 1):
                lo, hi = groups[g], groups[g + 1]
                c_lo, c_hi = int(chunk0[lo]), int(chunk0[hi])
                for c0 in range(c_lo, c_hi, step):
                    m = min(step, c_hi - c0)
                    _lib.check(_lib.lib().tt_gather_chunks(_ptr(clip_tab), _ptr(t_chunk0), n, c0, m, L, _ptr(batch), stream))
                    lat, skips = self._codes(batch[:m].view(m, 1, L))
                    for stage, reconstruct in zip(stages, (False, True)):
                        if stage is None:
                            continue
                        part = stage[c0 - c_lo:c0 - c_lo + m]
                        if fused:
                            self.decoder.last_stage_c8(lat, reconstruct, skips, out=part)
                        else:
                            y = self.decoder.forward_c8(lat, reconstruct, skips)
                            if self.HEAD_MODE is not None:          # both channels carry the head's output, as in _chunked
                                y = ops.channel0(y, self.HEAD_MODE).unsqueeze(-1).expand(-1, -1, -1, 2)
                            part.copy_(y)
                tab_g = ctypes.c_void_p(t_chunk0.data_ptr() + 4 * lo)
                max_chunks = int(chunks[lo:hi].max())
                for stage, reconstruct in zip(stages, (False, True)):
                    if stage is None:
                        continue
                    o = F * int(out0[lo])
                    if not reconstruct:
                        dst = (None, _ptr(trn[o:])) if as_act else (_ptr(trn[2 * o:]), None)
                    else:
                        coeffs = torch.empty((F * int(out0[hi] - out0[lo]), 2), **f32)
                        dst = (_ptr(coeffs), None)
                    if fused:
                        _lib.check(_lib.lib().tt_conv_out_crossfade_clips(_ptr(stage), _ptr(window), _ptr(w_out), _ptr(b_out), tab_g, hi - lo,
                                                                          c_hi - c_lo, max_chunks, self.decoder.channels[4], F, M, *dst, stream))
                    else:
                        _lib.check(_lib.lib().tt_chunk_crossfade_clips(_ptr(stage), _ptr(window), tab_g, hi - lo, max_chunks, F, M, *dst,
                                                                       stream))
                    if reconstruct:
                        _lib.check(_lib.lib().tt_cqt_inverse_clips(self.sliCQ._plan(device).handle, _ptr(coeffs),
                                                                   ctypes.c_void_p(t_block0.data_ptr() + 4 * lo), hi - lo,
                                                                   int(block0[hi] - block0[lo]), _ptr(audio[int(block0[lo]) * L:]),
                                                                   _ptr(peaks[lo:]), 1, stream))
            acts = wavs = None
            if want_transcription:
                if not as_act:
                    # a variant's own activation function, once over the whole buffer (element-wise: the same values as per clip)
                    pairs = self.to_activations(trn.view(1, 1, -1, 2).permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
                    trn = pairs.reshape(-1) if pairs.is_contiguous() else pairs.contiguous().reshape(-1)
                    acts = [trn[2 * F * a:2 * F * b].view(F, b - a, 2).permute(2, 0, 1) for a, b in zip(out0[:-1].tolist(), out0[1:].tolist())]
                else:
                    acts = [trn[F * a:F * b].view(F, b - a) for a, b in zip(out0[:-1].tolist(), out0[1:].tolist())]
            if want_reconstruction:
                wavs = [audio[L * a:L * b].view(1, L * (b - a)) for a, b in zip(block0[:-1].tolist(), block0[1:].tolist())]
            return acts, wavs

    # ---- one long clip over several GPUs (BASELINE.json configs[4]) ---------------------------------------------------
    # Blocks are independent except for the 50 % cross-fade with the two neighbouring chunks (modules.py:259-263): a rank that
    # owns output blocks [b0, b1) needs the audio of those blocks plus half a block on either side and nothing else - no
    # collective on the compute path; the results are all-gathered (and `reconstruct` shares one scalar MAX for the peak).
    def shard_audio(self, audio, rank, world):
        """(B, 1, N) -> (the rank's slice with its half-block halos, b0, b1): contiguous ranges of output blocks."""
        return shard_audio(self.sliCQ.pad_to_block_length(audio), self.sliCQ.block_length, rank, world)

    def transcribe_sharded(self, audio, group=None, rank=None, world=None, gather=True):
        """transcribe() of a clip every rank holds, each rank computing a contiguous range of blocks.  Returns the whole
        (B, F, T) activations on every rank (gather=True, via all_gather over `group`) or the rank's own frames."""
        group, rank, world = _resolve_group(group, rank, world)
        sub, b0, b1 = self.shard_audio(audio, rank, world)
        M, F = self.sliCQ.max_window_length, self.sliCQ.n_bins
        if b1 > b0:
            local = self._chunked(sub, True, False, prepadded=True)[0]
        else:
            local = torch.empty((audio.size(0), F, 0), dtype=torch.float32, device=audio.device)
        return _gather_frames(local, -1, M, audio, self.sliCQ.block_length, group, world) if gather else local

    def reconstruct_sharded(self, audio, group=None, rank=None, world=None, gather=True):
        """reconstruct() of a clip every rank holds, sharded like transcribe_sharded; the reference's global peak normalise
        (cqtwrapper.py:209-211) is one scalar MAX all-reduce over `group`."""
        group, rank, world = _resolve_group(group, rank, world)
        sub, b0, b1 = self.shard_audio(audio, rank, world)
        L = self.sliCQ.block_length
        if b1 > b0:
            rec = self._chunked(sub, False, True, prepadded=True)[1].permute(0, 3, 1, 2)
            local = self._decode_shared_peak(rec, group)
        else:
            local = torch.empty((audio.size(0), 1, 0), dtype=torch.float32, device=audio.device)
            if group is not None:                      # still take part in the peak exchange
                import torch.distributed as dist
                dist.all_reduce(torch.zeros(1, device=audio.device), op=dist.ReduceOp.MAX, group=group)
        return _gather_frames(local, -1, L, audio, L, group, world) if gather else local

    def transcribe_and_reconstruct_sharded(self, audio, group=None, rank=None, world=None, gather=True):
        """Both results for a clip every rank holds from ONE encoder pass per rank (transcribe_sharded + reconstruct_sharded run two)."""
        group, rank, world = _resolve_group(group, rank, world)
        sub, b0, b1 = self.shard_audio(audio, rank, world)
        M, F, L = self.sliCQ.max_window_length, self.sliCQ.n_bins, self.sliCQ.block_length
        if b1 > b0:
            act, rec = self._chunked(sub, True, True, prepadded=True)
            wav = self._decode_shared_peak(rec.permute(0, 3, 1, 2), group)
        else:
            act = torch.empty((audio.size(0), F, 0), dtype=torch.float32, device=audio.device)
            wav = torch.empty((audio.size(0), 1, 0), dtype=torch.float32, device=audio.device)
            if group is not None:
                import torch.distributed as dist
                dist.all_reduce(torch.zeros(1, device=audio.device), op=dist.ReduceOp.MAX, group=group)
        if not gather:
            return act, wav
        return _gather_frames(act, -1, M, audio, L, group, world), _gather_frames(wav, -1, L, audio, L, group, world)

    def forward(self, audio, consistency=False):
        """modules.py:338-393: audio (B, 1, N) -> (reconstruction, latents, transcription, transcription_rec, transcription_scr, {}), the
        last two None unless `consistency` (a bool or an int, as experiments/train.py passes it).

        In train mode with grad mode on, every layer runs through its autograd Function (framework/layer_grads.py) and the outputs carry
        the graph: the reference's loop body (`model(audio, consistency=True)`, `to_activations`, the objectives, `backward()`) trains
        the model.  The coefficient outputs are views of the internal interleaved pairs.  In eval mode or under no_grad this is inference:
        no graph, buffers reused.  Either way the model runs outside autocast (see _no_autocast)."""
        grad = self._graph()
        with _no_autocast(), torch.set_grad_enabled(grad):
            rec, trn, lat = self._passes(self._features(audio), grad)
            trn_rec = trn_scr = None
            if consistency:
                trn_rec, trn_scr, _ = self._passes(trn, grad)
                trn_rec, trn_scr = self._output(trn_rec, grad), self._output(trn_scr, grad)
            latents = P.from_c8(lat, self.encoder.latent_size).squeeze(-2)
            return self._output(rec, grad), latents, self._output(trn, grad), trn_rec, trn_scr, dict()

    # ---- full-track forward in time tiles (experiments/evaluate.py:81-95 feeds whole tracks through model(audio)) -------------------
    # Only the convolutions see across frames, and only +-1 frame (convin / convout) and +-6 frames per block of three dilated
    # residual stages: +-25 frames per encoder or decoder pass, +-50 for the outputs of forward(), +-100 for the consistency pair.
    TILE_HALO = 128

    def forward_tiled(self, audio, consistency=False, tile_frames=32768):
        """
        TimbreTrap.forward (modules.py:338-393) on a track of any length with bounded activation memory: the CQT runs over the whole
        track (blocks are independent), the encoder / decoder passes over tiles of `tile_frames` frames plus TILE_HALO frames of true
        context on either side, of which only the tile's own frames are kept.  Same outputs as forward(), bit for bit
        (tests/test_model_gpu.py::test_forward_tiled_equals_untiled).
        """
        if tile_frames % 128 or tile_frames <= 0:
            raise ValueError('tile_frames must be a positive multiple of 128')
        with torch.no_grad():
            feats = self._features(audio)                                   # (B, F, T, 2)
            B, F, T, _ = feats.shape
            h = self.TILE_HALO
            n_out = 2 if self.HEAD_MODE is None else 1
            outs = [torch.empty((B, n_out, F, T), dtype=torch.float32, device=feats.device) for _ in range(4 if consistency else 2)]
            latents = torch.empty((B, self.encoder.latent_size, T), dtype=torch.float32, device=feats.device)
            for t0 in range(0, T, tile_frames):
                t1 = min(T, t0 + tile_frames)
                a, b = max(0, t0 - h), min(T, t1 + h)
                keep = slice(t0 - a, t0 - a + (t1 - t0))
                rec, trn, lat = self._passes(feats[:, :, a:b].contiguous())
                tile = [rec, trn] + (list(self._passes(trn)[:2]) if consistency else [])
                for out, y in zip(outs, tile):
                    out[..., t0:t1] = y.permute(0, 3, 1, 2)[:, :n_out, ..., keep]     # a variant's output is channel 0 of its pairs
                latents[..., t0:t1] = P.from_c8(lat, self.encoder.latent_size).squeeze(-2)[..., keep]
        return outs[0], latents, outs[1], (outs[2] if consistency else None), (outs[3] if consistency else None), dict()


class FiLM(nn.Module):
    """modules.py:842-889: y = x * gamma(condition) + beta(condition) per latent channel.  Parameter holder here - the layer is folded
    into the packed weights / bias table of decoder.convin (packing.pack_deconv_in_film); `forward` is the reference arithmetic on
    whatever device the tensors live (a (B, D, T) latent tensor, cheap) for callers that use the layer on its own."""

    def __init__(self, embedding_size, n_conditions):
        super().__init__()
        self.gamma = nn.Linear(n_conditions, embedding_size)
        self.beta = nn.Linear(n_conditions, embedding_size)

    def forward(self, x, condition):
        return (x.transpose(-1, -2) * self.gamma(condition) + self.beta(condition)).transpose(-1, -2)


class TimbreTrapFiLM(TimbreTrap):
    """modules.py:780-840: the switch is a FiLM layer on the latents instead of an indicator channel.  `latent_size` must be given
    (the reference's `latent_size=None` branch reads `nn.Sequential.in_channels`, which does not exist, modules.py:799)."""

    def __init__(self, sample_rate, n_octaves, bins_per_octave, secs_per_block=3, latent_size=None, model_complexity=1, skip_connections=False):
        TimbreTrap.__init__(self, sample_rate, n_octaves, bins_per_octave, secs_per_block, latent_size, model_complexity, skip_connections)
        if latent_size is None:
            raise ValueError('TimbreTrapFiLM needs an explicit latent_size (so does the reference: modules.py:799 fails without one)')
        old = self.decoder.convin[0]
        self.decoder.convin = nn.Sequential(nn.ConvTranspose2d(latent_size, old.out_channels, kernel_size=old.kernel_size), nn.ELU(inplace=True))
        self.film_layer = FiLM(latent_size, n_conditions=2)
        # not a registered sub-module of the decoder (state_dict keys stay the reference's: film_layer.* at the top level only)
        object.__setattr__(self.decoder, '_film', self.film_layer)

    def __setstate__(self, state):
        super().__setstate__(state)
        object.__setattr__(self.decoder, '_film', self.film_layer)


class TimbreTrapMag(TimbreTrap):
    """modules.py:892-1001: magnitude-CQT variant - one-channel encoder input |c|, one-channel relu output, tanh activations."""

    HEAD_MODE = 1               # relu (modules.py:976)
    ACTIVATIONS_MODE = 3        # tanh (modules.py:996): tanh(relu(h)) = tanh(h) on the head's output h >= 0

    def __init__(self, sample_rate, n_octaves, bins_per_octave, secs_per_block=3, latent_size=None, model_complexity=1, skip_connections=False):
        TimbreTrap.__init__(self, sample_rate, n_octaves, bins_per_octave, secs_per_block, latent_size, model_complexity, skip_connections)
        c0 = self.encoder.convin[0].out_channels
        cl = self.decoder.convout.in_channels
        self.encoder.convin = nn.Sequential(nn.Conv2d(1, c0, kernel_size=3, padding='same'), nn.ELU(inplace=True))
        self.decoder.convout = nn.Conv2d(cl, 1, kernel_size=3, padding='same')

    def _features(self, audio):
        """modules.py:947: to_magnitude(sliCQ(audio)) as pairs (|c|, 0)."""
        return ops.widen(CQT._magnitude(self.sliCQ.encode_interleaved(audio).permute(0, 3, 1, 2), False))

    def to_activations(self, coefficients):
        """modules.py:980-1001: tanh of the (B, 1, F, T) magnitude coefficients -> (B, F, T), differentiable when grad mode is on and the
        coefficients require grad.  Like the reference's `squeeze(-3)`, a two-channel tensor (what the inherited chunk loop produces for
        this variant) keeps its channel axis."""
        _lib.require_cuda(coefficients, 'coefficients')
        return torch.tanh(coefficients.float().squeeze(-3))


class TimbreTrapMagDB(TimbreTrapMag):
    """modules.py:1004-1075: decibel-magnitude variant - encoder input to_decibels(|c|) in [0, 1], sigmoid output, activations = output."""

    HEAD_MODE = 2               # sigmoid (modules.py:1052)
    ACTIVATIONS_MODE = 0        # the head's output as it is (modules.py:1056-1075)

    def _features(self, audio):
        """modules.py:1024-1027."""
        mag = CQT._magnitude(self.sliCQ.encode_interleaved(audio).permute(0, 3, 1, 2), False)
        return ops.widen(CQT.to_decibels(mag))

    def to_activations(self, coefficients):
        """modules.py:1056-1075: the sigmoid output as it is (a view; gradients pass straight through)."""
        return coefficients.squeeze(-3)
