"""
Thin torch-tensor wrappers over the conv and element-wise entry points of the C ABI (include/timbre_trap_b200.h).
Tensors are C8 planar bf16 (B, CG, H, T, 8) unless noted; weights are already packed (packing.py).
PyTorch is used for allocation and stream ownership only.
"""

import torch

from .. import _lib


def _check_c8(x, name='x'):
    _lib.require_cuda(x, name)
    if x.dtype != torch.bfloat16 or x.dim() != 5 or x.size(-1) != 8 or not x.is_contiguous():
        raise ValueError(f'{name} must be a contiguous C8 planar bf16 tensor (B, CG, H, T, 8), got {tuple(x.shape)} {x.dtype}')


def conv_lat(x, w, b, latent_pad):
    _check_c8(x)
    B, CG, H, T, _ = x.shape
    y = torch.empty((B, latent_pad // 8, 1, T, 8), dtype=torch.bfloat16, device=x.device)
    _lib.launch('tt_conv_lat', x, y, w, b, B, CG * 8, H, latent_pad, T)
    return y


def deconv_in(lat, w, bias_table, c0_pad, h0, act=True):
    _check_c8(lat, 'latents')
    B, CG, _, T, _ = lat.shape
    y = torch.empty((B, c0_pad // 8, h0, T, 8), dtype=torch.bfloat16, device=lat.device)
    _lib.launch('tt_deconv_in', lat, y, w, bias_table, B, CG * 8, c0_pad, h0, T, int(act))
    return y


def conv_in(coeffs_bft2, w, b, c0, packed4=False, act=True):
    """coeffs (B, F, T, 2) fp32 interleaved -> C8 planar (B, 1, F, T, 8), or the packed 4-channel layout (B, F, T, 4).  act=False
    (packed output only): without the ELU - the data gradient of Decoder.convout."""
    _lib.require_cuda(coeffs_bft2, 'coefficients')
    if not (act or packed4):
        raise ValueError('conv_in without the ELU writes the packed 4-channel layout only (pass packed4=True)')
    B, F, T, _ = coeffs_bft2.shape
    y = torch.empty((B, F, T, 4) if packed4 else (B, 1, F, T, 8), dtype=torch.bfloat16, device=coeffs_bft2.device)
    _lib.launch('tt_conv_in', coeffs_bft2, y, w, b, B, c0, F, T, int(packed4) if act else 2)
    return y


def conv_out(x, w, b, c):
    """C8 planar (B, 1, F, T, 8) or packed 4-channel (B, F, T, 4) -> coeffs (B, F, T, 2) fp32 interleaved."""
    packed4 = x.dim() == 4
    if packed4:
        _check_p4(x)
        B, F, T, _ = x.shape
    else:
        _check_c8(x)
        B, _, F, T, _ = x.shape
    y = torch.empty((B, F, T, 2), dtype=torch.float32, device=x.device)
    _lib.launch('tt_conv_out', x, y, w, b, B, c, F, T, int(packed4))
    return y


def _check_p4(x, name='x'):
    _lib.require_cuda(x, name)
    if x.dtype != torch.bfloat16 or x.dim() != 4 or x.size(-1) != 4 or x.size(-2) % 2 or not x.is_contiguous():
        raise ValueError(f'{name} must be a contiguous packed 4-channel bf16 tensor (B, H, T, 4) with even T, got {tuple(x.shape)} {x.dtype}')


def res_block_rs(x, w1, w2, bias, c_real, dilation, out=None, fold=False, mid_out=None):
    """Row-stationary fused residual block (csrc/res_rs.cu).  x C8 planar: weights from packing.pack_res_rs, or with fold=True
    (C <= 8, even T) packing.pack_res_rs_fold(..., fold=2); x packed 4-channel (B, H, T, 4): packing.pack_res_rs_pairs, or with
    fold=True (T % 4 == 0) packing.pack_res_rs_fold(..., fold=4)."""
    packed4 = x.dim() == 4
    if packed4:
        _check_p4(x)
        B, H, T, _ = x.shape
        C, c_real = 8, min(c_real, 4)
        layout = 4 if fold else 1
    else:
        _check_c8(x)
        B, CG, H, T, _ = x.shape
        C = CG * 8
        layout = 2 if fold else 0
    _lib.require_cuda(bias, 'bias')
    y = torch.empty_like(x) if out is None else out
    if mid_out is None:
        _lib.launch('tt_res_block_rs', x, y, w1, w2, bias, B, C, c_real, H, T, dilation, layout)
    else:
        # the inner activation ELU(W1 * x + b1) as well, in the layout of y (kept by the loss step for its backward pass)
        if mid_out.shape != y.shape or mid_out.dtype != y.dtype or not mid_out.is_contiguous():
            raise ValueError('mid_out must be a contiguous tensor of the shape and dtype of the output')
        _lib.launch('tt_res_block_rs_mid', x, y, mid_out, w1, w2, bias, B, C, c_real, H, T, dilation, layout)
    return y


def conv_down_strip(x, w, cout_pad, act=True):
    """C8 planar input, or the packed 4-channel layout (B, H, T, 4) with weights from packing.pack_down_pairs (4 -> 8 channels)."""
    packed4 = x.dim() == 4
    if packed4:
        _check_p4(x)
        B, H, T, _ = x.shape
        cin = 8
    else:
        _check_c8(x)
        B, CG, H, T, _ = x.shape
        cin = CG * 8
    y = torch.empty((B, cout_pad // 8, (H - 4) // 2 + 1, T, 8), dtype=torch.bfloat16, device=x.device)
    _lib.launch('tt_conv_down_strip', x, y, w, B, cin, cout_pad, H, T, int(packed4), int(act))
    return y


def conv_up_strip(x, w, cout_pad, out_pad, packed4_out=False, act=True):
    _check_c8(x)
    B, CG, H, T, _ = x.shape
    Hout = 2 * H + 2 + out_pad
    y = torch.empty((B, Hout, T, 4) if packed4_out else (B, cout_pad // 8, Hout, T, 8), dtype=torch.bfloat16, device=x.device)
    _lib.launch('tt_conv_up_strip', x, y, w, B, CG * 8, cout_pad, H, out_pad, T, int(packed4_out), int(act))
    return y


def conv_same(x, w, bias, k, dilation=1, act=False, times_elu_grad_of=None, plus=None):
    """3x3 dilated 'same' conv (k = 3) or 1x1 conv (k = 1) on a C8 planar tensor, optional ELU (tile kernel, tensor cores).  Fused
    epilogues of the residual blocks' backward: `times_elu_grad_of=a` multiplies by ELU'(.) given the activated tensor a, `plus=g` adds g."""
    _check_c8(x)
    B, CG, H, T, _ = x.shape
    y = torch.empty_like(x)
    post, e = (1, times_elu_grad_of) if times_elu_grad_of is not None else ((2, plus) if plus is not None else (0, None))
    if e is not None and (e.shape != x.shape or e.dtype != x.dtype or not e.is_contiguous()):
        raise ValueError('the post-op tensor must have the shape, dtype and (contiguous) layout of the output')
    _lib.launch('tt_conv_same_post', x, y, w, bias, B, CG * 8, H, T, k, dilation, int(act), post, e)
    return y


def widen(x):
    """(B, F, T) fp32 -> interleaved (B, F, T, 2) pairs (x, 0) (tt_widen_pairs)."""
    x = x.detach().float().contiguous()
    out = torch.empty(tuple(x.shape) + (2,), dtype=torch.float32, device=x.device)
    if x.numel():
        _lib.launch('tt_widen_pairs', x, x.numel(), out)
    return out


def channel0(pairs, mode):
    """interleaved (B, F, T, 2) -> (B, F, T): channel 0 through a non-linearity (tt_channel0_activation modes)."""
    out = torch.empty(pairs.shape[:-1], dtype=torch.float32, device=pairs.device)
    if out.numel():
        _lib.launch('tt_channel0_activation', pairs, out.numel(), mode, out)
    return out


def add_scaled(x, e, scale, out=None):
    """x + scale * e on two bf16 tensors of one layout, one pass (tt_add_scaled_bf16); scale is a 0-dim device tensor."""
    if x.shape != e.shape or x.dtype != torch.bfloat16 or e.dtype != torch.bfloat16:
        raise ValueError(f'skip connection: {tuple(x.shape)} {x.dtype} vs {tuple(e.shape)} {e.dtype}')
    out = torch.empty_like(x) if out is None else out
    s = scale.detach().float().reshape(1)
    _lib.launch('tt_add_scaled_bf16', x, e.contiguous(), s, out, x.numel())
    return out
