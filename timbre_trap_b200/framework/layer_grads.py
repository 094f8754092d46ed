"""
The layers of the model as torch.autograd.Functions (the model runs them with `forward_c8(..., grad=True)`, framework/modules.py),
and the head and activation Functions (the loss Functions are in framework/objectives.py).

Each layer's forward is the inference kernel, handed in by the module as a closure; its backward stays in the bf16 inference layouts
(C8 planar / packed 4-channel): weight gradients are tcgen05 GEMMs over the pixel axis with a fixed-order reduction (csrc/wgrad_tc.cu),
data gradients are the forward kernels on transformed weights without activation, and ELU derivatives, skip connections and
re-layouts are one-pass bf16 kernels.  A layer computes its weight and bias gradients only when autograd asks for them
(`ctx.needs_input_grad`): the weight-gradient launch of a layer whose parameters are all frozen is skipped.  PyTorch's autograd engine only
walks the graph and accumulates `.grad`; there is no cuDNN / ATen compute on the path.
"""

import torch
from torch.utils.weak import WeakIdKeyDictionary

from .. import _lib
from . import ops
from . import packing as P
from .cqt import CQT
from .packing import _PackedCache


# ---- residual blocks: the whole backward in the inference layouts (bf16), convolutions AND weight gradients on the tensor cores ----
def _ew(fn_name, *tensors):
    """element-wise bf16 kernel over tensors of one common layout -> new tensor like the first"""
    out = torch.empty_like(tensors[0])
    _lib.launch(fn_name, *tensors, out, out.numel())
    return out


def _as_c8(t):
    """packed 4-channel (B, H, T, 4) -> C8 planar (B, 1, H, T, 8) (native re-layout kernel); C8 tensors pass through"""
    if t.dim() == 5:
        return t
    B, H, T, _ = t.shape
    out = torch.empty((B, 1, H, T, 8), dtype=torch.bfloat16, device=t.device)
    _lib.launch('tt_p4_to_c8', t, out, B * H * T)
    return out


def _to_layout_of(c8, ref):
    """C8 planar (B, 1, H, T, 8) -> the layout of `ref` (packed 4-channel or C8)"""
    if ref.dim() == 5:
        return c8
    out = torch.empty_like(ref)
    _lib.launch('tt_c8_to_p4', c8, out, out.numel() // 4)
    return out


_WGRAD_SCRATCH = {}
# weight tensor -> {tag: (stamp, packed)}: one entry per (weight, tag), dropped with the weight
_BW_PACKS = WeakIdKeyDictionary()


def _scratch(pool, device, n):
    """One growing fp32 scratch buffer per device (the weight-gradient partials): reused by every layer, reallocated only to grow."""
    buf = pool.get(device)
    if buf is None or buf.numel() < n:
        buf = torch.empty(n, dtype=torch.float32, device=device)
        pool[device] = buf
    return buf


def _bw_pack(weight, tag, build, deps=()):
    """Packed (kernel-layout) weights of the backward pass, built once per optimisation step per layer: the same layer runs backward
    two to four times per step (two encoder, four decoder passes), and every pack is a handful of tiny launches.  One entry per
    (weight, tag), rebuilt in place when the weight or one of `deps` (other tensors the pack is built from) has been modified - a torch
    optimizer's in-place update bumps the version counter, TrainStep's AdamW kernel bumps _PackedCache.epoch - or moved."""
    stamp = (_PackedCache.epoch,) + tuple((t.data_ptr(), t._version) for t in (weight,) + tuple(deps))
    packs = _BW_PACKS.get(weight)
    if packs is None:
        packs = _BW_PACKS[weight] = {}
    hit = packs.get(tag)
    if hit is None or hit[0] != stamp:
        with torch.no_grad():
            hit = packs[tag] = (stamp, build())
    return hit[1]


def _bw_pack_entries():
    """Number of packs held (one per (weight, tag))."""
    return sum(len(v) for v in _BW_PACKS.values())


def _wgrad_same(x8, dz8, cin, cout, k, d):
    """(dW (cout, cin, k, k), db (cout)) fp32 of a 'same' conv from C8 planar bf16 x and dz (tt_conv_wgrad_same, tensor cores)."""
    B, CGi, H, T, _ = x8.shape
    scratch = _scratch(_WGRAD_SCRATCH, x8.device, int(_lib.lib().tt_wgrad_scratch_floats(B, H, T)))
    dw = torch.zeros((cout, cin, k, k), dtype=torch.float32, device=x8.device)
    db = torch.zeros(cout, dtype=torch.float32, device=x8.device)
    _lib.launch('tt_conv_wgrad_same', x8, dz8, dw, db, B, CGi * 8, dz8.size(1) * 8, cin, cout, H, T, k, d, scratch)
    return dw, db


class _ResFn(torch.autograd.Function):
    """ResidualConv2dBlock: fused forward kernel, which also writes the inner activation ELU(W1 * x + b1) it stages in shared memory
    (tt_res_block_rs_mid) - the backward needs it and a recompute costs a whole 3x3 conv launch per block; the backward stays in bf16
    C8 planar end to end - both data-gradient convolutions through the tile kernel (tt_conv_same_post), both weight gradients through the
    MN-major tcgen05 kernels (tt_conv_wgrad_same), the ELU derivatives / residual add as one-pass element-wise kernels."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, run, c, d):
        a1 = torch.empty_like(x)
        y = run(x, a1)
        ctx.save_for_backward(x, y, a1, w1, b1, w2)
        ctx.meta = (c, d)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, y, a1, w1, b1, w2 = ctx.saved_tensors
        c, d = ctx.meta
        need = ctx.needs_input_grad
        gy = gy.contiguous()
        dz2 = _as_c8(_ew('tt_res_out_bwd_bf16', gy, y, x))                       # gy * ELU'(z2), activated 1x1 output = y - x
        a1 = _as_c8(a1)                                                          # the inner activation, as the forward staged it
        dw1 = db1 = dw2 = db2 = gx = None
        if need[3] or need[4]:
            dw2, db2 = _wgrad_same(a1, dz2, c, c, 1, 1)
        if not (need[0] or need[1] or need[2]):
            return gx, dw1, db1, _needed(dw2, need[3]), _needed(db2, need[4]), None, None, None
        w2_t = _bw_pack(w2, 'res1x1T', lambda: P.pack_res1x1(w2.detach().float().transpose(0, 1).contiguous()))
        dz1 = ops.conv_same(dz2, w2_t, None, 1, 1, times_elu_grad_of=a1)         # W2^T dz2, times ELU'(z1): one launch
        if need[1] or need[2]:
            dw1, db1 = _wgrad_same(_as_c8(x), dz1, c, c, 3, d)
        if need[0]:
            w1_t = _bw_pack(w1, 'res3x3T', lambda: P.pack_res3x3(w1.detach().float().transpose(0, 1).flip(2, 3).contiguous()))
            if gy.dim() == 5:
                gx = ops.conv_same(dz1, w1_t, None, 3, d, plus=gy)               # gx = gy + W1^T (*) dz1: the residual add in the epilogue
            else:
                gx = _to_layout_of(ops.conv_same(dz1, w1_t, None, 3, d), x)      # packed 4-channel stage: re-layout, then add
                gx = ops.add_scaled(gy, gx, torch.ones((), dtype=torch.float32, device=gx.device), out=gx)
        return gx, _needed(dw1, need[1]), _needed(db1, need[2]), _needed(dw2, need[3]), _needed(db2, need[4]), None, None, None


def _needed(g, flag):
    """A gradient that one weight-gradient launch produced together with another: handed back only where autograd asked for it."""
    return g if flag else None


def _wgrad_updown(fine8, coarse8, cfine, ccoarse, transposed):
    """Weight / bias gradients of a (4,1) stride-(2,1) layer from C8 planar bf16 tensors (tt_conv_wgrad_updown, tensor cores):
    sconv: (fine = layer input, coarse = dz) -> dW (ccoarse, cfine, 4, 1), db (ccoarse); tconv (transposed): (fine = dz, coarse = layer
    input) -> dW (ccoarse, cfine, 4, 1) in the ConvTranspose2d layout, db (cfine)."""
    B, CGf, Hf, T, _ = fine8.shape
    Hc = coarse8.size(2)
    scratch = _scratch(_WGRAD_SCRATCH, fine8.device, int(_lib.lib().tt_wgrad_scratch_floats(B, Hc, T)))
    dw = torch.zeros((ccoarse, cfine, 4, 1), dtype=torch.float32, device=fine8.device)
    db = torch.zeros(cfine if transposed else ccoarse, dtype=torch.float32, device=fine8.device)
    _lib.launch('tt_conv_wgrad_updown', fine8, coarse8, dw, db, B, CGf * 8, coarse8.size(1) * 8, cfine, ccoarse, Hf, Hc, T, int(transposed),
                scratch)
    return dw, db


class _DownFn(torch.autograd.Function):
    """EncoderBlock.sconv + ELU (modules.py:626-629).  Backward in the inference layouts: ELU derivative (element-wise), weight gradient
    (tensor-core GEMM over the pixel axis), data gradient = the transposed-conv forward kernel without activation on W seen as a
    ConvTranspose2d weight (in = Cout, out = Cin)."""

    @staticmethod
    def forward(ctx, x, weight, bias, run, cin, cout):
        y = run(x)
        ctx.save_for_backward(x, y, weight)
        ctx.meta = (cin, cout)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, y, weight = ctx.saved_tensors
        cin, cout = ctx.meta
        need = ctx.needs_input_grad
        dz = _ew('tt_elu_bwd_bf16', gy.contiguous(), y)
        x8 = _as_c8(x)
        dw = db = gx = None
        if need[1] or need[2]:
            dw, db = _wgrad_updown(x8, dz, cin, cout, False)
        if need[0]:
            hin, hout = x8.size(2), dz.size(2)
            wt = _bw_pack(weight, 'downT', lambda: P.pack_up_strip(weight.detach().float(), torch.zeros(cin, device=weight.device)))
            gx = ops.conv_up_strip(dz, wt, P.pad8(cin), hin - 2 * hout - 2, packed4_out=x.dim() == 4, act=False)
        return gx, _needed(dw, need[1]), _needed(db, need[2]), None, None, None


class _UpFn(torch.autograd.Function):
    """DecoderBlock.tconv + ELU (modules.py:685-688).  Backward: data gradient = the strided-conv forward kernel without activation on
    W^T seen as a Conv2d weight (out = Cin, in = Cout)."""

    @staticmethod
    def forward(ctx, x, weight, bias, run, cin, cout):
        y = run(x)
        ctx.save_for_backward(x, y, weight)
        ctx.meta = (cin, cout)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, y, weight = ctx.saved_tensors
        cin, cout = ctx.meta
        need = ctx.needs_input_grad
        dz = _ew('tt_elu_bwd_bf16', gy.contiguous(), y)                          # layout of y (packed 4-channel for the last stage)
        dw = db = gx = None
        if need[1] or need[2]:
            dw, db = _wgrad_updown(_as_c8(dz), x, cout, cin, True)
        if need[0]:
            # ConvTranspose2d (cin, cout, 4, 1) read as a Conv2d weight (out = cin, in = cout)
            pack = P.pack_down_pairs if dz.dim() == 4 else P.pack_down_strip
            wd = _bw_pack(weight, 'upT', lambda: pack(weight.detach().float().contiguous(), torch.zeros(cin, device=weight.device)))
            gx = ops.conv_down_strip(dz, wd, P.pad8(cin), act=False)
        return gx, _needed(dw, need[1]), _needed(db, need[2]), None, None, None


_LAT_SCRATCH = {}


def _wgrad_lat(tall8, flat8, ctall, cflat, dw, db, row_sums):
    """tt_conv_wgrad_lat: accumulates into dw (cflat.., ctall, H, 1) [first cflat rows], db (cflat) and row_sums (ctall, H) (either may be None).
    The kernel takes up to 128 flat-side channels; wider latents go through it in slices of 128 (a slice of the 1-row latents is a tiny copy)."""
    B, CGt, H, T, _ = tall8.shape
    scratch = _scratch(_LAT_SCRATCH, tall8.device, int(_lib.lib().tt_wgrad_lat_scratch_floats(B, H, T)))
    for c0 in range(0, cflat, 128):
        c1 = min(cflat, c0 + 128)
        flat = flat8[:, c0 // 8:c0 // 8 + 16].contiguous()
        _lib.launch('tt_conv_wgrad_lat', tall8, flat, dw[c0:c1], None if db is None else db[c0:c1], row_sums if c0 == 0 else None,
                    B, CGt * 8, flat.size(1) * 8, ctall, c1 - c0, H, T, scratch)


class _LatFn(torch.autograd.Function):
    """Encoder.convlat (modules.py:446, no activation).  Backward in the inference layouts: weight gradient = tap-grouped tensor-core GEMM
    over (b, t); data gradient = the Decoder.convin forward kernel (a (H, 1) transposed conv) without activation on the same weights."""

    @staticmethod
    def forward(ctx, x, weight, bias, run, c4, d, d_pad):
        y = run(x)
        ctx.save_for_backward(x, weight)
        ctx.meta = (c4, d, d_pad)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        c4, d, d_pad = ctx.meta
        need = ctx.needs_input_grad
        gy = gy.contiguous()
        dw = db = gx = None
        if need[1] or need[2]:
            dw = torch.zeros(weight.shape, dtype=torch.float32, device=x.device)
            db = torch.zeros(d, dtype=torch.float32, device=x.device)
            _wgrad_lat(x, gy, c4, d, dw, db, None)
        if need[0]:
            # gx[ci, h, t] = sum_co W[co, ci, h] gy[co, t]: ConvTranspose2d with weight (in = co, out = ci, H, 1)
            w, table = _bw_pack(weight, 'latT', lambda: P.pack_deconv_in_film(weight.detach().float(), torch.zeros(c4, device=x.device),
                                                                              torch.ones(d, device=x.device), torch.zeros(d, device=x.device), d_pad))
            gx = ops.deconv_in(gy, w, table, P.pad8(c4), x.size(2), act=False)
        return gx, _needed(dw, need[1]), _needed(db, need[2]), None, None, None, None


def _pairs_to_c8(pairs):
    """fp32 interleaved (B, F, T, 2) -> C8 planar bf16 (B, 1, F, T, 8) (tt_pairs_to_c8)."""
    pairs = pairs.contiguous()
    B, F_, T, _ = pairs.shape
    out = torch.empty((B, 1, F_, T, 8), dtype=torch.bfloat16, device=pairs.device)
    _lib.launch('tt_pairs_to_c8', pairs, B * F_ * T, out)
    return out


def _two_channels(w, dim):
    """A one-channel conv weight of the magnitude variants zero-padded to two channels along `dim`, as the forward packs run it
    (Encoder._packed / Decoder._packed); two-channel weights pass through."""
    if w.size(dim) == 2:
        return w
    return torch.cat((w, torch.zeros_like(w)), dim=dim)


class _InFn(torch.autograd.Function):
    """Encoder.convin + ELU (modules.py:430-433) with a packed 4-channel output.  Backward: ELU derivative on the packed tensor; weight
    gradient on the tensor cores (both operands re-laid out to C8 planar bf16 by one-pass kernels); data gradient (only the consistency
    pass asks for it) = the Decoder.convout forward kernel on transposed, flipped weights.  The one-channel convin of the magnitude
    variants (modules.py:908-911) reads pairs (x, 0) against zero-padded weights: its weight gradient is the first input column of the
    two-channel one."""

    @staticmethod
    def forward(ctx, coeffs, weight, bias, run, c0):
        y = run(coeffs)
        ctx.save_for_backward(coeffs, y, weight)
        ctx.c0 = c0
        return y

    @staticmethod
    def backward(ctx, gy):
        coeffs, y, weight = ctx.saved_tensors
        c0 = ctx.c0
        need = ctx.needs_input_grad
        dz = _ew('tt_elu_bwd_bf16', gy.contiguous(), y)
        dw = db = gx = None
        if need[1] or need[2]:
            dw, db = _wgrad_same(_pairs_to_c8(coeffs), _as_c8(dz), 2, c0, 3, 1)
            if weight.size(1) == 1:
                dw = dw[:, :1]
        if need[0]:
            wt, zb = _bw_pack(weight, 'inT', lambda: (_two_channels(weight.detach().float(), 1).transpose(0, 1).flip(2, 3).contiguous(),  # (2, c0, 3, 3)
                                                      torch.zeros(2, device=dz.device)))
            gx = ops.conv_out(dz, wt, zb, c0)
        return gx, _needed(dw, need[1]), _needed(db, need[2]), None, None


class _OutFn(torch.autograd.Function):
    """Decoder.convout (modules.py:543, no activation) on a packed 4-channel input.  Backward: weight gradient on the tensor cores;
    data gradient = the Encoder.convin forward kernel without ELU on transposed, flipped weights.  The one-channel convout of the
    magnitude variants (modules.py:913) runs as two channels with a zero second one: its gradients are the first rows of the
    two-channel ones."""

    @staticmethod
    def forward(ctx, x, weight, bias, run, c):
        y = run(x)
        ctx.save_for_backward(x, weight)
        ctx.c = c
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        c = ctx.c
        need = ctx.needs_input_grad
        gy = gy.contiguous()
        dw = db = gx = None
        if need[1] or need[2]:
            dw, db = _wgrad_same(_as_c8(x), _pairs_to_c8(gy), c, 2, 3, 1)
            if weight.size(0) == 1:
                dw, db = dw[:1], db[:1]
        if need[0]:
            wt, zb = _bw_pack(weight, 'outT', lambda: (_two_channels(weight.detach().float(), 0).transpose(0, 1).flip(2, 3).contiguous(),  # (c, 2, 3, 3)
                                                       torch.zeros(c, device=gy.device)))
            gx = ops.conv_in(gy, wt, zb, c, packed4=True, act=False)
        return gx, _needed(dw, need[1]), _needed(db, need[2]), None, None


class _SkipAddFn(torch.autograd.Function):
    """Decoder skip connection (modules.py:568-589) with TimbreTrap.apply_skip_connections' learnable weight (:110-112):
    out = x + w * e on two bf16 tensors of one layout, one pass; gradients: x <- g, e <- w * g (one pass), w <- <g, e> (deterministic)."""

    @staticmethod
    def forward(ctx, x, e, w):
        scale = w.detach().float().reshape(1)
        ctx.save_for_backward(e, scale)
        return ops.add_scaled(x, e, scale)

    @staticmethod
    def backward(ctx, g):
        e, scale = ctx.saved_tensors
        g = g.contiguous()
        ge = gw = None
        if ctx.needs_input_grad[1]:
            ge = ops.add_scaled(g, g, scale - 1.0)                                   # g + (w - 1) g = w g
        if ctx.needs_input_grad[2]:
            gw = torch.empty((), dtype=torch.float32, device=g.device)
            scratch = torch.empty(int(_lib.lib().tt_dot_scratch_floats()), dtype=torch.float32, device=g.device)
            _lib.launch('tt_dot_bf16', g, e, g.numel(), gw, scratch)
        return g, ge, gw


class _ActivationsFn(torch.autograd.Function):
    """TimbreTrap.to_activations (modules.py:271-289) on interleaved coefficients (B, F, T, 2) -> (B, F, T)."""

    @staticmethod
    def forward(ctx, coeffs):
        ctx.save_for_backward(coeffs)
        return CQT._magnitude(coeffs.permute(0, 3, 1, 2), True)

    @staticmethod
    def backward(ctx, gact):
        (coeffs,) = ctx.saved_tensors
        g = torch.empty_like(coeffs)
        _lib.launch('tt_activations_bwd', coeffs, gact.contiguous(), g, gact.numel())
        return g


def _channel0_bwd(pairs, gpairs, mode):
    """(g * f'(v0), 0) for the pre-activation pairs v and the output-pair gradient g (tt_channel0_activation_bwd)."""
    gpairs = gpairs.contiguous()
    g = torch.empty_like(pairs)
    _lib.launch('tt_channel0_activation_bwd', pairs, gpairs, pairs.numel() // 2, mode, g)
    return g


class _HeadFn(torch.autograd.Function):
    """The output head of the magnitude variants on the decoder's pairs (modules.py:976, 1052): (B, F, T, 2) -> pairs (f(v0), 0),
    f = relu (mode 1) or sigmoid (mode 2); the one-channel output stays a pair with a zero second channel."""

    @staticmethod
    def forward(ctx, pairs, mode):
        ctx.save_for_backward(pairs)
        ctx.mode = mode
        return ops.widen(ops.channel0(pairs, mode))

    @staticmethod
    def backward(ctx, g):
        (pairs,) = ctx.saved_tensors
        return _channel0_bwd(pairs, g, ctx.mode), None


class _Channel0ActivationsFn(torch.autograd.Function):
    """to_activations of the magnitude variants on the head's pairs (h, 0) -> (B, F, T): tanh(h) for TimbreTrapMag (modules.py:996;
    mode 3, tanh(relu(h)) = tanh(h) as h >= 0), h for TimbreTrapMagDB (:1056-1075; mode 0)."""

    @staticmethod
    def forward(ctx, pairs, mode):
        ctx.save_for_backward(pairs)
        ctx.mode = mode
        return ops.channel0(pairs, mode)

    @staticmethod
    def backward(ctx, gact):
        (pairs,) = ctx.saved_tensors
        return _channel0_bwd(pairs, ops.widen(gact), ctx.mode), None


class _IndicatorFn(torch.autograd.Function):
    """
    Decoder.convin on latents + the constant indicator channel (modules.py:139-142, 533-536).  Forward: tt_deconv_in with the
    indicator folded into the bias table.  Backward: transposed-conv gradients with the indicator channel written out (its weight
    row receives a gradient, its input does not).
    """

    @staticmethod
    def forward(ctx, lat, weight, bias, run, flag, d, c0):
        y = run(lat)
        ctx.save_for_backward(lat, y, weight)
        ctx.meta = (flag, d, c0)
        return y

    @staticmethod
    def backward(ctx, gy):
        lat, y, weight = ctx.saved_tensors
        flag, d, c0 = ctx.meta
        need = ctx.needs_input_grad
        # ELU derivative, tap-grouped tensor-core weight gradient (rows 0 .. D-1; the indicator row and the bias are row sums of dz),
        # data gradient = the Encoder.convlat forward kernel on the first D weight rows
        dz = _ew('tt_elu_bwd_bf16', gy.contiguous(), y)
        dw = db = glat = None
        if need[1] or need[2]:
            h0 = y.size(2)
            dw = torch.zeros(weight.shape, dtype=torch.float32, device=lat.device)
            rows = torch.zeros((c0, h0), dtype=torch.float32, device=lat.device)
            _wgrad_lat(dz, lat, c0, d, dw, None, rows)
            dw[d, :, :, 0] = flag * rows
            db = rows.sum(dim=1)
        if need[0]:
            d_pad = lat.size(1) * 8
            wl, zl = _bw_pack(weight, 'decinT', lambda: (P.pack_lat(weight.detach().float()[:d], d_pad), torch.zeros(d_pad, device=lat.device)))
            glat = ops.conv_lat(dz, wl, zl, d_pad)
        return glat, _needed(dw, need[1]), _needed(db, need[2]), None, None, None, None


class _FiLMConvInFn(torch.autograd.Function):
    """
    TimbreTrapFiLM: the FiLM layer and Decoder.convin (modules.py:801-809, 838-840), y = ELU(convT(gamma * z + beta)) with gamma / beta
    = film_layer.gamma / .beta of the one-hot condition [transcribe, not transcribe] (`hot` = the column of its 1).  Forward:
    tt_deconv_in on the folded pack (packing.pack_deconv_in_film).  Backward: ELU derivative; the tensor-core sums G = dz x z and the
    row sums of dz (tt_conv_wgrad_lat); every parameter gradient from those in one launch (tt_film_convin_grad); latent gradient =
    the Encoder.convlat forward kernel on W scaled by gamma.
    """

    @staticmethod
    def forward(ctx, lat, weight, bias, gamma_w, gamma_b, beta_w, beta_b, run, hot, d, c0):
        y = run(lat)
        ctx.save_for_backward(lat, y, weight, gamma_w, gamma_b, beta_w, beta_b)
        ctx.meta = (hot, d, c0)
        return y

    @staticmethod
    def backward(ctx, gy):
        lat, y, weight, gamma_w, gamma_b, beta_w, beta_b = ctx.saved_tensors
        hot, d, c0 = ctx.meta
        need = ctx.needs_input_grad
        dz = _ew('tt_elu_bwd_bf16', gy.contiguous(), y)
        grads = _film_convin_grads(dz, lat, weight, gamma_w, gamma_b, beta_w, beta_b, hot, d, c0, params=any(need[1:7]), latents=need[0])
        return tuple(_needed(g, n) for g, n in zip(grads, need[:7])) + (None,) * 4


def _film_convin_grads(dz, lat, weight, gamma_w, gamma_b, beta_w, beta_b, hot, d, c0, params=True, latents=True):
    """Gradients of _FiLMConvInFn from dz (C8 planar, after the ELU derivative) and the latents lat (C8 planar, H = 1):
    (latents (bf16, C8), convin weight, convin bias, gamma.weight, gamma.bias, beta.weight, beta.bias); `params` / `latents` False:
    the six parameter gradients (one weight-gradient and one FiLM launch) / the latent gradient are skipped and come back None."""
    h0 = dz.size(2)
    dev = lat.device
    dw = db = dgw = dgb = dbw = dbb = glat = None
    if params:
        G = torch.zeros(weight.shape, dtype=torch.float32, device=dev)
        rows = torch.zeros((c0, h0), dtype=torch.float32, device=dev)
        _wgrad_lat(dz, lat, c0, d, G, None, rows)
        dw = torch.empty_like(G)
        db = torch.empty(c0, dtype=torch.float32, device=dev)
        dgw, dbw = torch.empty_like(gamma_w), torch.empty_like(beta_w)
        dgb, dbb = torch.empty_like(gamma_b), torch.empty_like(beta_b)
        _lib.launch('tt_film_convin_grad', G, rows, weight, gamma_w, gamma_b, beta_w, beta_b, d, c0, h0, hot, dw, db, dgw, dgb, dbw, dbb)
    if latents:
        d_pad = lat.size(1) * 8

        def build():
            gamma = gamma_w.detach()[:, hot] + gamma_b.detach()                          # film_layer.gamma(one-hot cond)
            return P.pack_lat(weight.detach().float() * gamma.view(-1, 1, 1, 1), d_pad), torch.zeros(d_pad, device=dev)
        # gamma differs between the two passes (the tag) and depends on the FiLM parameters (rebuilt when they change)
        wl, zl = _bw_pack(weight, ('filmT', hot), build, deps=(gamma_w, gamma_b))
        glat = ops.conv_lat(dz, wl, zl, d_pad)
    return glat, dw, db, dgw, dgb, dbw, dbb
