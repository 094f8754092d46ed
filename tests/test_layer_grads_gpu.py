"""
One layer's backward at a time: every autograd Function of framework/layer_grads.py, called on its own with the run closure and the
packed weights its module builds, against float64 torch autograd of the same layer written as the reference writes it
(oracle/model_ref.py's _res, _enc_block, _dec_block, encoder_ref, decoder_ref).  The input is a leaf in the layer's internal layout
(C8 planar or packed 4-channel bf16); the reference forward gets the bf16-rounded input and the bf16-rounded weights the tensor-core
kernels multiply (Encoder.convin and Decoder.convout run in fp32 on the CUDA cores: their reference keeps fp32 weights), and its
gradient is taken with respect to the fp32 parameter.  Shapes are those the model produces: the BASE geometry (22.05 kHz, 9 x 60
bins, model_complexity 2: heights 540 / 269 / 133 / 65 / 31, T = 1024 frames per 3 s block) and the SMALL test geometry
(model_complexity 1: 72 / 35 / 16 / 7 / 2).

Every input, weight and bias gradient is gated on its own: rel-L2, max-abs over max|want| and, for tensors with image rows, the
worst row's rel-L2 (a wrong edge, seam or output_padding row that the whole-tensor norm averages away).  The pad lanes of every data
gradient must be exactly zero (tt_dot_bf16 and the bias sums read whole tensors), and two backward passes must agree bit for bit.
The element-wise backward kernels are checked bit-exactly against their fp32 formulas.
"""
from collections import namedtuple

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

Gate = namedtuple('Gate', 'rel max row', defaults=(None,))

# Gates: about twice the worst value measured over a layer's cases on a B200 (bf16 activations and activation gradients; the
# weight-gradient sums in fp32).  Every data gradient: rel-L2 2.1e-3, max-abs 4.1e-3 of max|want|, worst row 2.2e-3.
DATA_GATE = Gate(4.5e-3, 8e-3, 4.5e-3)


@pytest.fixture
def force_strip_rows():
    """tt_set_strip_rows(rows) for the duration of one test (automatic split restored afterwards)."""
    from timbre_trap_b200 import _lib
    yield lambda rows: _lib.check(_lib.lib().tt_set_strip_rows(rows))
    _lib.lib().tt_set_strip_rows(0)


def _randn(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(shape, generator=g) * scale


def _bf(x):
    return x.to(torch.bfloat16).float()


def _q(w):
    """bf16 rounding of a float64 leaf that autograd passes straight through: the gradient lands on the unrounded parameter."""
    return w.to(torch.bfloat16).to(torch.float64)


def _leaf(p):
    return p.detach().cpu().double().requires_grad_(True)


def _to(x, layout):
    """(B, C, H, T) -> the internal layout on the GPU: 'p4' packed 4-channel (B, H, T, 4), 'c8' C8 planar (B, CG, H, T, 8)."""
    from timbre_trap_b200.framework import packing as P
    return (P.to_p4(x) if layout == 'p4' else P.to_c8(x)).cuda()


def _from(t, C):
    from timbre_trap_b200.framework import packing as P
    return (P.from_p4(t, C) if t.dim() == 4 else P.from_c8(t, C)).cpu().double()


def _pad_lanes(t, C):
    """The channels >= C of an internal-layout tensor (what the layer does not have)."""
    if t.dim() == 4:
        return t[..., C:]
    B, CG, H, T, _ = t.shape
    return t.permute(0, 1, 4, 2, 3).reshape(B, CG * 8, H, T)[:, C:]


def _grads(y, inputs, gy):
    """Input and parameter gradients of y . gy, twice on the same graph: the backward is deterministic bit for bit."""
    first = torch.autograd.grad(y, inputs, gy, retain_graph=True)
    again = torch.autograd.grad(y, inputs, gy, retain_graph=True)
    for i, (a, b) in enumerate(zip(first, again)):
        assert torch.equal(a, b), f'gradient {i} differs between two backward passes'
    return first


def _check(tag, name, got, want, gate, row_dim=None):
    got, want = got.detach().cpu().double(), want.detach().cpu().double()
    assert got.shape == want.shape, (tag, name, tuple(got.shape), tuple(want.shape))
    d = got - want
    rel = float(d.norm() / want.norm())
    mx = float(d.abs().max() / want.abs().max())
    row = None
    if row_dim is not None:
        rows_d = d.movedim(row_dim, 0).reshape(d.size(row_dim), -1).norm(dim=1)
        rows_w = want.movedim(row_dim, 0).reshape(d.size(row_dim), -1).norm(dim=1)
        row = float((rows_d / rows_w.clamp_min(1e-300)).max())
    print(f'grad-err {tag} {name}: rel-L2 {rel:.2e} max {mx:.2e}' + ('' if row is None else f' worst row {row:.2e}'))
    assert rel <= gate.rel, (tag, name, 'rel-L2', rel)
    assert mx <= gate.max, (tag, name, 'max-abs', mx)
    assert row is None or row <= gate.row, (tag, name, 'worst row', row)


# ---- ResidualConv2dBlock (_ResFn) -----------------------------------------------------------------------------------------------
# measured: weights 5.7e-3 rel-L2 / 5.6e-3 max; biases 1.9e-2 / 2.2e-2, the 2-channel block at H = 2 (a sum over 1024 pixels that
# nearly cancels; 8.9e-3 at the model's heights).  Inputs of std 4: weights 7.3e-3 / 8.1e-3, biases 8.4e-3 / 7.8e-3, data unchanged.
RES_GATES = dict(weight=Gate(1.2e-2, 1.2e-2), bias=Gate(4e-2, 4.5e-2))
RES_LARGE_GATES = dict(weight=Gate(1.5e-2, 1.6e-2), bias=Gate(1.7e-2, 1.6e-2))

# (C, H, T, layout): the forward picks fold4 (packed, T % 4 == 0), pairs (packed, T % 4 == 2), fold2 (C8, C <= 8, even T) or planar
RES_CASES = [(4, 540, 1024, 'p4'), (8, 269, 1024, 'c8'), (16, 133, 1024, 'c8'), (32, 65, 1024, 'c8'),     # BASE, model_complexity 2
             (16, 133, 200, 'c8'),                                                                         # T not a multiple of 128
             (2, 72, 258, 'p4'), (4, 35, 200, 'c8'), (8, 16, 131, 'c8'), (16, 7, 200, 'c8'),               # SMALL, model_complexity 1
             (2, 2, 256, 'p4'), (8, 3, 130, 'c8'), (32, 2, 128, 'c8')]                                     # H <= 2d


def _res_case(C, H, T, layout, d, x_std=1.0, gates=RES_GATES):
    from timbre_trap_b200.framework.modules import ResidualConv2dBlock
    seed = C * 1000 + H * 10 + d
    torch.manual_seed(seed)
    blk = ResidualConv2dBlock(C, C, kernel_size=3, dilation=d)
    blk.packed4 = layout == 'p4'
    blk = blk.cuda()
    B = 1 if T >= 1024 else 2
    x0 = _bf(_randn((B, C, H, T), seed + 1, x_std))
    g0 = _bf(_randn((B, C, H, T), seed + 2))
    x = _to(x0, layout).requires_grad_(True)
    c1, c2 = blk.conv1[0], blk.conv2[0]
    params = [c1.weight, c1.bias, c2.weight, c2.bias]
    y = blk.forward_c8(x, grad=True)
    got = _grads(y, [x] + params, _to(g0, layout))

    xr = x0.double().requires_grad_(True)
    pr = [_leaf(p) for p in params]
    a1 = F.elu(F.conv2d(xr, _q(pr[0]), pr[1], padding=d, dilation=d))
    yr = xr + F.elu(F.conv2d(a1, _q(pr[2]), pr[3]))
    want = torch.autograd.grad(yr, [xr] + pr, g0.double())

    tag = f'res C={C} H={H} T={T} {layout} d={d} std={x_std}'
    _check(tag, 'x', _from(got[0], C), want[0], DATA_GATE, row_dim=2)
    for name, g, w in zip(('conv1.weight', 'conv1.bias', 'conv2.weight', 'conv2.bias'), got[1:], want[1:]):
        _check(tag, name, g, w, gates[name.split('.')[1]])
    pad = _pad_lanes(got[0], C)
    assert pad.numel() == 0 or float(pad.float().abs().max()) == 0.0, 'non-zero pad lanes in the input gradient'


@pytest.mark.parametrize('C,H,T,layout', RES_CASES)
@pytest.mark.parametrize('d', [1, 2, 3])
def test_residual_block_backward(C, H, T, layout, d):
    """_ResFn: tt_res_out_bwd_bf16, the 1x1 data gradient with ELU'(z1) in its epilogue, the 3x3 data gradient with the residual add
    in its epilogue (C8) or through tt_c8_to_p4 + tt_add_scaled_bf16 (packed), both tensor-core weight gradients."""
    _res_case(C, H, T, layout, d)


@pytest.mark.parametrize('C,H,T,layout', [(4, 540, 1024, 'p4'), (16, 133, 1024, 'c8')])
def test_residual_block_backward_large_inputs(C, H, T, layout):
    """Inputs of std 4: the backward recovers ELU'(z2) from y - x, both bf16, so its error grows with |x| - measured on a B200 at
    about 2x (weights) and 2x - 5x (biases) the std-1 figures of the same shapes; the data gradient 2.1e-3 against 1.8e-3."""
    _res_case(C, H, T, layout, 1, x_std=4.0, gates=RES_LARGE_GATES)


def test_residual_block_backward_strip_seams(force_strip_rows):
    """Forced 7-row strips: seams inside the forward and both data-gradient convolutions."""
    force_strip_rows(7)
    _res_case(8, 269, 1024, 'c8', 2)


# ---- EncoderBlock.sconv (_DownFn) and DecoderBlock.tconv (_UpFn) --------------------------------------------------------------
# measured: weights 2.7e-3 rel-L2 / 3.4e-3 max, biases 2.3e-3 / 2.5e-3
UPDOWN_GATES = dict(weight=Gate(5.5e-3, 7e-3), bias=Gate(5e-3, 5.5e-3))


def _down_case(cin, cout, H, T, layout):
    from timbre_trap_b200.framework import layer_grads as LG, ops, packing as P
    from timbre_trap_b200.framework.modules import EncoderBlock
    seed = cin * 1000 + H
    torch.manual_seed(seed)
    blk = EncoderBlock(cin, cout).cuda()
    c = blk.sconv[0]
    pack = P.pack_down_pairs if layout == 'p4' else P.pack_down_strip

    def run(t):
        return ops.conv_down_strip(t, pack(c.weight, c.bias), P.pad8(cout))
    B = 1 if T >= 1024 else 2
    x0 = _bf(_randn((B, cin, H, T), seed + 1))
    x = _to(x0, layout).requires_grad_(True)
    y = LG._DownFn.apply(x, c.weight, c.bias, run, cin, cout)
    g0 = _bf(_randn((B, cout, y.size(2), T), seed + 2))
    got = _grads(y, [x, c.weight, c.bias], _to(g0, 'c8'))

    xr = x0.double().requires_grad_(True)
    pr = [_leaf(c.weight), _leaf(c.bias)]
    yr = F.elu(F.conv2d(xr, _q(pr[0]), pr[1], stride=(2, 1)))
    want = torch.autograd.grad(yr, [xr] + pr, g0.double())

    tag = f'down {cin}->{cout} H={H} T={T} {layout}'
    _check(tag, 'x', _from(got[0], cin), want[0], DATA_GATE, row_dim=2)
    _check(tag, 'weight', got[1], want[1], UPDOWN_GATES['weight'])
    _check(tag, 'bias', got[2], want[2], UPDOWN_GATES['bias'])
    pad = _pad_lanes(got[0], cin)
    assert pad.numel() == 0 or float(pad.float().abs().max()) == 0.0, 'non-zero pad lanes in the input gradient'


# (cin, cout, H, T, layout); the data gradient is tt_conv_up_strip without ELU, output_padding = H % 2
DOWN_CASES = [(4, 8, 540, 1024, 'p4'), (8, 16, 269, 1024, 'c8'), (16, 32, 133, 1024, 'c8'), (32, 64, 65, 1024, 'c8'),    # BASE
              (32, 64, 65, 200, 'c8'),
              (2, 4, 72, 200, 'p4'), (4, 8, 35, 200, 'c8'), (8, 16, 16, 200, 'c8'), (16, 32, 7, 200, 'c8'),              # SMALL
              (2, 4, 37, 256, 'p4')]                                                                                     # odd, packed


@pytest.mark.parametrize('cin,cout,H,T,layout', DOWN_CASES)
def test_strided_conv_backward(cin, cout, H, T, layout):
    """_DownFn: tt_elu_bwd_bf16, tt_conv_wgrad_updown, data gradient through the linear epilogue of tt_conv_up_strip (packed output
    for the packed first stage); both input-height parities."""
    _down_case(cin, cout, H, T, layout)


def test_strided_conv_backward_strip_seams(force_strip_rows):
    force_strip_rows(5)
    _down_case(8, 16, 269, 1024, 'c8')


def _up_case(cin, cout, H, op, T, packed):
    from timbre_trap_b200.framework import layer_grads as LG, ops, packing as P
    from timbre_trap_b200.framework.modules import DecoderBlock
    seed = cin * 1000 + H * 10 + op
    torch.manual_seed(seed)
    blk = DecoderBlock(cin, cout, padding=op).cuda()
    c = blk.tconv[0]

    def run(t):
        return ops.conv_up_strip(t, P.pack_up_strip(c.weight, c.bias), P.pad8(cout), op, packed4_out=packed)
    B = 1 if T >= 1024 else 2
    x0 = _bf(_randn((B, cin, H, T), seed + 1))
    x = _to(x0, 'c8').requires_grad_(True)
    y = LG._UpFn.apply(x, c.weight, c.bias, run, cin, cout)
    Hout = 2 * H + 2 + op
    g0 = _bf(_randn((B, cout, Hout, T), seed + 2))
    got = _grads(y, [x, c.weight, c.bias], _to(g0, 'p4' if packed else 'c8'))

    xr = x0.double().requires_grad_(True)
    pr = [_leaf(c.weight), _leaf(c.bias)]
    yr = F.elu(F.conv_transpose2d(xr, _q(pr[0]), pr[1], stride=(2, 1), output_padding=(op, 0)))
    want = torch.autograd.grad(yr, [xr] + pr, g0.double())

    tag = f'up {cin}->{cout} H={H} op={op} T={T} packed={packed}'
    _check(tag, 'x', _from(got[0], cin), want[0], DATA_GATE, row_dim=2)
    _check(tag, 'weight', got[1], want[1], UPDOWN_GATES['weight'])
    _check(tag, 'bias', got[2], want[2], UPDOWN_GATES['bias'])
    pad = _pad_lanes(got[0], cin)
    assert pad.numel() == 0 or float(pad.float().abs().max()) == 0.0, 'non-zero pad lanes in the input gradient'


# (cin, cout, H, output_padding, T, packed output); the data gradient is tt_conv_down_strip without ELU
UP_CASES = [(64, 32, 31, 1, 1024, False), (32, 16, 65, 1, 1024, False), (16, 8, 133, 1, 1024, False), (8, 4, 269, 0, 1024, True),  # BASE
            (16, 8, 133, 1, 200, False),
            (32, 16, 2, 1, 200, False), (16, 8, 7, 0, 200, False), (8, 4, 16, 1, 200, False), (4, 2, 35, 0, 200, True),           # SMALL
            (4, 2, 17, 1, 256, True), (64, 32, 31, 0, 256, False)]


@pytest.mark.parametrize('cin,cout,H,op,T,packed', UP_CASES)
def test_transposed_conv_backward(cin, cout, H, op, T, packed):
    """_UpFn: tt_elu_bwd_bf16 (packed output for the last stage), tt_conv_wgrad_updown (transposed), data gradient through the
    linear epilogue of tt_conv_down_strip; output_padding 0 and 1."""
    _up_case(cin, cout, H, op, T, packed)


def test_transposed_conv_backward_strip_seams(force_strip_rows):
    force_strip_rows(3)
    _up_case(32, 16, 65, 1, 1024, False)


# ---- Encoder.convlat (_LatFn) and Decoder.convin with the indicator channel (_IndicatorFn) -------------------------------------
# measured: weights 2.0e-3 rel-L2 / 3.8e-3 max / 2.1e-3 worst row; biases 7.8e-8 (convlat: fp32 sums of bf16 values) and 2.0e-3
# (Decoder.convin: sums of the bf16 ELU derivative)
LAT_WEIGHT_GATE = Gate(4.5e-3, 8e-3, 4.5e-3)
LAT_CASES = [(c4, h4, d) for c4 in (32, 64) for h4 in (2, 31) for d in (24, 40, 128, 200)]    # latents padded to 32, 64, 128, 256


@pytest.mark.parametrize('C4,H4,D', LAT_CASES)
def test_latent_conv_backward(C4, H4, D):
    """_LatFn: tt_conv_wgrad_lat (two slices of 128 latent channels for D = 200), data gradient through tt_deconv_in without ELU."""
    from timbre_trap_b200.framework import layer_grads as LG, ops, packing as P
    from timbre_trap_b200.framework.modules import _latent_pad
    seed = C4 * 1000 + H4 * 10 + D
    torch.manual_seed(seed)
    conv = nn.Conv2d(C4, D, kernel_size=(H4, 1)).cuda()
    d_pad = _latent_pad(D)

    def run(t):
        return ops.conv_lat(t, P.pack_lat(conv.weight, d_pad), P.pad_vec(conv.bias, d_pad), d_pad)
    T = 1024 if H4 == 31 else 200
    B = 1 if T >= 1024 else 2
    x0 = _bf(_randn((B, C4, H4, T), seed + 1))
    x = _to(x0, 'c8').requires_grad_(True)
    y = LG._LatFn.apply(x, conv.weight, conv.bias, run, C4, D, d_pad)
    g0 = _bf(_randn((B, D, 1, T), seed + 2))
    got = _grads(y, [x, conv.weight, conv.bias], _to(F.pad(g0, (0, 0, 0, 0, 0, d_pad - D)), 'c8'))

    xr = x0.double().requires_grad_(True)
    pr = [_leaf(conv.weight), _leaf(conv.bias)]
    yr = F.conv2d(xr, _q(pr[0]), pr[1])
    want = torch.autograd.grad(yr, [xr] + pr, g0.double())

    tag = f'lat C4={C4} H4={H4} D={D}'
    _check(tag, 'x', _from(got[0], C4), want[0], DATA_GATE, row_dim=2)
    _check(tag, 'weight', got[1], want[1], LAT_WEIGHT_GATE, row_dim=2)
    _check(tag, 'bias', got[2], want[2], Gate(1.5e-7, 1.5e-7))


@pytest.mark.parametrize('C0,H0,D', LAT_CASES)
@pytest.mark.parametrize('flag', [0, 1])
def test_decoder_convin_backward(C0, H0, D, flag):
    """_IndicatorFn: tt_elu_bwd_bf16, tt_conv_wgrad_lat with the row sums that are the indicator row's and the bias's gradients, latent
    gradient through tt_conv_lat on the first D weight rows; indicator 0 (transcribe: its weight row gets no gradient) and 1."""
    from timbre_trap_b200.framework import layer_grads as LG, ops, packing as P
    from timbre_trap_b200.framework.modules import _latent_pad
    seed = C0 * 1000 + H0 * 10 + D + flag
    torch.manual_seed(seed)
    ct = nn.ConvTranspose2d(D + 1, C0, kernel_size=(H0, 1)).cuda()
    d_pad = _latent_pad(D)
    w_pack, tables = P.pack_deconv_in(ct.weight, ct.bias, d_pad)

    def run(t):
        return ops.deconv_in(t, w_pack, tables[flag].contiguous(), P.pad8(C0), H0)
    T = 1024 if H0 == 31 else 200
    B = 1 if T >= 1024 else 2
    z0 = _bf(_randn((B, D, 1, T), seed + 1))
    lat = _to(F.pad(z0, (0, 0, 0, 0, 0, d_pad - D)), 'c8').requires_grad_(True)
    y = LG._IndicatorFn.apply(lat, ct.weight, ct.bias, run, float(flag), D, C0)
    g0 = _bf(_randn((B, C0, H0, T), seed + 2))
    got = _grads(y, [lat, ct.weight, ct.bias], _to(g0, 'c8'))

    zr = z0.double().requires_grad_(True)
    pr = [_leaf(ct.weight), _leaf(ct.bias)]
    full = torch.cat((zr, torch.full_like(zr[:, :1], float(flag))), dim=1)
    w = torch.cat((_q(pr[0][:D]), pr[0][D:]))                      # the indicator row is folded into the fp32 bias table
    yr = F.elu(F.conv_transpose2d(full, w, pr[1]))
    want = torch.autograd.grad(yr, [zr] + pr, g0.double())

    tag = f'convin C0={C0} H0={H0} D={D} flag={flag}'
    _check(tag, 'latents', _from(got[0], D), want[0], DATA_GATE)
    _check(tag, 'weight', got[1], want[1], LAT_WEIGHT_GATE, row_dim=2)
    _check(tag, 'bias', got[2], want[2], Gate(3e-3, 4.5e-3))
    if flag:
        _check(tag, 'indicator row', got[1][D], want[1][D], Gate(3e-3, 4.5e-3))
    else:
        assert float(got[1][D].abs().max()) == 0.0
    pad = _pad_lanes(got[0], D)
    assert pad.numel() == 0 or float(pad.float().abs().max()) == 0.0, 'non-zero pad lanes in the latent gradient'


# ---- Encoder.convin (_InFn) and Decoder.convout (_OutFn) ------------------------------------------------------------------------
# measured: Encoder.convin coefficients 1.3e-3 rel-L2 / 1.7e-3 max / 1.5e-3 worst row, weights 2.7e-3 / 2.5e-3, biases 1.5e-3 / 2.1e-3;
# Decoder.convout input 1.7e-3 / 3.1e-3 / 1.8e-3, weights and biases 1.4e-6 (bf16 x bf16 products, fp32 sums)
IN_GATES = dict(data=Gate(3e-3, 3.5e-3, 3e-3), weight=Gate(5.5e-3, 5.5e-3), bias=Gate(3e-3, 4.5e-3))
OUT_GATES = dict(data=Gate(3.5e-3, 6.5e-3, 4e-3), weight=Gate(2.5e-6, 2.5e-6), bias=Gate(3e-6, 3e-6))
INOUT_CASES = [(4, 540, 1024), (2, 72, 200), (4, 72, 260)]


@pytest.mark.parametrize('C0,F_,T', INOUT_CASES)
@pytest.mark.parametrize('n_in', [2, 1])
def test_encoder_convin_backward(C0, F_, T, n_in):
    """_InFn: two input channels, and the one channel (x, 0) of the magnitude variants; ELU derivative on the packed output,
    tt_pairs_to_c8 + tensor-core weight gradient, data gradient through tt_conv_out on the transposed, flipped weights."""
    from timbre_trap_b200.framework import layer_grads as LG, ops
    seed = C0 * 1000 + F_ + n_in
    torch.manual_seed(seed)
    conv = nn.Conv2d(n_in, C0, kernel_size=3, padding=1).cuda()
    w_in = conv.weight.detach().float()
    if n_in == 1:
        w_in = torch.cat((w_in, torch.zeros_like(w_in)), dim=1)

    def run(t):
        return ops.conv_in(t, w_in.contiguous(), conv.bias.detach().float().contiguous(), C0, packed4=True)
    B = 1 if T >= 1024 else 2
    x0 = _randn((B, n_in, F_, T), seed + 1)
    pairs = x0.permute(0, 2, 3, 1)
    if n_in == 1:
        pairs = torch.cat((pairs, torch.zeros_like(pairs)), dim=-1)
    coeffs = pairs.contiguous().cuda().requires_grad_(True)
    y = LG._InFn.apply(coeffs, conv.weight, conv.bias, run, C0)
    g0 = _bf(_randn((B, C0, F_, T), seed + 2))
    got = _grads(y, [coeffs, conv.weight, conv.bias], _to(g0, 'p4'))

    xr = x0.double().requires_grad_(True)
    pr = [_leaf(conv.weight), _leaf(conv.bias)]
    yr = F.elu(F.conv2d(xr, pr[0], pr[1], padding=1))
    want = torch.autograd.grad(yr, [xr] + pr, g0.double())

    tag = f'convin C0={C0} F={F_} T={T} n_in={n_in}'
    gx = got[0].cpu().double()
    _check(tag, 'coefficients', gx[..., :n_in].permute(0, 3, 1, 2), want[0], IN_GATES['data'], row_dim=2)
    if n_in == 1:
        assert float(gx[..., 1].abs().max()) == 0.0, 'gradient into the zero channel of the one-channel pairs'
    _check(tag, 'weight', got[1], want[1], IN_GATES['weight'])
    _check(tag, 'bias', got[2], want[2], IN_GATES['bias'])


@pytest.mark.parametrize('C,F_,T', INOUT_CASES)
@pytest.mark.parametrize('n_out', [2, 1])
def test_decoder_convout_backward(C, F_, T, n_out):
    """_OutFn: tt_pairs_to_c8 + tensor-core weight gradient, data gradient through tt_conv_in with packed4=2 (packed output, no ELU)."""
    from timbre_trap_b200.framework import layer_grads as LG, ops
    seed = C * 1000 + F_ + n_out
    torch.manual_seed(seed)
    conv = nn.Conv2d(C, n_out, kernel_size=3, padding=1).cuda()
    w_out, b_out = conv.weight.detach().float(), conv.bias.detach().float()
    if n_out == 1:
        w_out, b_out = torch.cat((w_out, torch.zeros_like(w_out))), torch.cat((b_out, torch.zeros_like(b_out)))

    def run(t):
        return ops.conv_out(t, w_out.contiguous(), b_out.contiguous(), C)
    B = 1 if T >= 1024 else 2
    x0 = _bf(_randn((B, C, F_, T), seed + 1))
    x = _to(x0, 'p4').requires_grad_(True)
    y = LG._OutFn.apply(x, conv.weight, conv.bias, run, C)
    g0 = _bf(_randn((B, n_out, F_, T), seed + 2))
    gy = g0.permute(0, 2, 3, 1)
    if n_out == 1:                                                   # the magnitude head hands back (g f'(v0), 0)
        gy = torch.cat((gy, torch.zeros_like(gy)), dim=-1)
    got = _grads(y, [x, conv.weight, conv.bias], gy.contiguous().cuda())

    xr = x0.double().requires_grad_(True)
    pr = [_leaf(conv.weight), _leaf(conv.bias)]
    yr = F.conv2d(xr, pr[0], pr[1], padding=1)
    want = torch.autograd.grad(yr, [xr] + pr, g0.double())

    tag = f'convout C={C} F={F_} T={T} n_out={n_out}'
    _check(tag, 'x', _from(got[0], C), want[0], OUT_GATES['data'], row_dim=2)
    _check(tag, 'weight', got[1], want[1], OUT_GATES['weight'])
    _check(tag, 'bias', got[2], want[2], OUT_GATES['bias'])
    pad = _pad_lanes(got[0], C)
    assert pad.numel() == 0 or float(pad.float().abs().max()) == 0.0, 'non-zero pad lanes in the input gradient'


# ---- skip connections (_SkipAddFn) ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('C,H,T,layout', [(16, 133, 1024, 'c8'), (4, 35, 200, 'c8'), (32, 65, 200, 'c8'), (4, 540, 1024, 'p4'),
                                          (2, 72, 200, 'p4')])
def test_skip_add_backward(C, H, T, layout):
    """out = x + w e: x <- g (the same tensor), e <- w g (one bf16 rounding of the fp32 product), w <- <g, e> (fp32, fixed order)."""
    from timbre_trap_b200.framework import layer_grads as LG
    seed = C * 1000 + H
    B = 1 if T >= 1024 else 2
    x0, e0, g0 = (_bf(_randn((B, C, H, T), seed + i)) for i in range(3))
    x = _to(x0, layout).requires_grad_(True)
    e = _to(e0, layout).requires_grad_(True)
    w = torch.tensor(0.8, device='cuda', requires_grad=True)
    out = LG._SkipAddFn.apply(x, e, w)
    g = _to(g0, layout)
    gx, ge, gw = _grads(out, [x, e, w], g)
    assert torch.equal(gx, g)
    want_e = (0.8 * g0.double())
    d = (_from(ge, C) - want_e).abs()
    assert bool((d <= (2 ** -8 + 1e-6) * want_e.abs()).all()), float(d.max())   # one bf16 rounding (half an ulp: <= 2^-8 relative)
    want_w = float((g0.double() * e0.double()).sum())
    assert abs(float(gw) - want_w) <= 1e-5 * float((g0.double() * e0.double()).abs().sum()), (float(gw), want_w)
    pad = _pad_lanes(ge, C)
    assert pad.numel() == 0 or float(pad.float().abs().max()) == 0.0


# ---- element-wise backward kernels ----------------------------------------------------------------------------------------------
def _bits(t):
    return t.contiguous().view(torch.int16).cpu()


def _special(t):
    """bf16 tensor with exact 0 and -1 in the first two sixteenths of its values."""
    flat = t.view(-1)
    k = flat.numel() // 16
    flat[:k] = 0.0
    flat[k:2 * k] = -1.0
    return t


def test_elu_bwd_bit_exact():
    """tt_elu_bwd_bf16: bf16(gy * (a > 0 ? 1 : a + 1)) in fp32, bit for bit, over a grid-stride loop; ELU'(0) = 1, ELU'(-1) = 0."""
    from timbre_trap_b200.framework import layer_grads as LG
    shape = (2, 2, 269, 1024, 8)
    gy = _randn(shape, 1).to(torch.bfloat16)
    a = _special(_randn(shape, 2).to(torch.bfloat16))
    got = LG._ew('tt_elu_bwd_bf16', gy.cuda(), a.cuda())
    af = a.float()
    want = (gy.float() * torch.where(af > 0, torch.ones_like(af), af + 1)).to(torch.bfloat16)
    assert torch.equal(_bits(got), _bits(want))


def test_res_out_bwd_bit_exact():
    """tt_res_out_bwd_bf16: bf16(gy * ELU'(y - x)) with y - x in fp32, bit for bit; y - x exactly 0 and exactly -1 included."""
    from timbre_trap_b200.framework import layer_grads as LG
    shape = (2, 2, 269, 1024, 8)
    gy = _randn(shape, 3).to(torch.bfloat16)
    x = (_randn(shape, 4) * 4).to(torch.bfloat16)
    y = (x.float() + F.elu(_randn(shape, 5))).to(torch.bfloat16)
    k = gy.numel() // 16
    y.view(-1)[:k] = x.view(-1)[:k]                                       # y - x = 0: ELU' = 1
    x.view(-1)[k:2 * k] = 0.25
    y.view(-1)[k:2 * k] = -0.75                                          # y - x = -1: ELU' = 0
    got = LG._ew('tt_res_out_bwd_bf16', gy.cuda(), y.cuda(), x.cuda())
    dz = y.float() - x.float()
    want = (gy.float() * torch.where(dz > 0, torch.ones_like(dz), dz + 1)).to(torch.bfloat16)
    assert torch.equal(_bits(got), _bits(want))


def test_p4_c8_round_trip():
    """tt_p4_to_c8 writes the 4 channels and zeros in lanes 4..7; tt_c8_to_p4 drops lanes 4..7: an exact round trip."""
    from timbre_trap_b200.framework import layer_grads as LG
    p4 = _randn((2, 269, 1024, 4), 6).to(torch.bfloat16).cuda()
    c8 = LG._as_c8(p4)
    assert c8.shape == (2, 1, 269, 1024, 8)
    assert torch.equal(_bits(c8[:, 0, ..., :4]), _bits(p4)) and float(c8[..., 4:].float().abs().max()) == 0.0
    c8[..., 4:] = 1.0                                                   # lanes 4..7 are not part of the packed layout
    back = LG._to_layout_of(c8, p4)
    assert back.shape == p4.shape and torch.equal(_bits(back), _bits(p4))


def test_pairs_to_c8_rounding():
    """tt_pairs_to_c8: round-to-nearest-even to bf16 (ties included), channels 2..7 zero."""
    from timbre_trap_b200.framework import layer_grads as LG
    pairs = _randn((2, 72, 200, 2), 7)
    ties = torch.tensor([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 2 ** -20 * (1 + 2 ** -8), 3.0 + 2 ** -7])
    pairs.view(-1)[:ties.numel()] = ties
    got = LG._pairs_to_c8(pairs.cuda())
    assert got.shape == (2, 1, 72, 200, 8)
    assert torch.equal(_bits(got[:, 0, ..., :2]), _bits(pairs.to(torch.bfloat16)))
    assert float(got[..., 2:].float().abs().max()) == 0.0


@pytest.mark.parametrize('n', [8, 3_000_000])
def test_dot_bf16_abi(n):
    """tt_dot_bf16 (the skip weights' gradient), called through the C ABI, against an fp64 sum: 8 values, and more than one
    grid-stride span (1184 CTAs x 256 threads x 8 values); the fixed-order reduction is bit-reproducible."""
    from timbre_trap_b200 import _lib
    a = (1 + 0.5 * _randn((n,), 8)).to(torch.bfloat16)
    b = (1 + 0.5 * _randn((n,), 9)).to(torch.bfloat16)
    lib = _lib.lib()
    scratch = torch.empty(int(lib.tt_dot_scratch_floats()), dtype=torch.float32, device='cuda')
    out = [torch.empty((), dtype=torch.float32, device='cuda') for _ in range(2)]
    ac, bc = a.cuda(), b.cuda()
    for o in out:
        _lib.check(lib.tt_dot_bf16(ac.data_ptr(), bc.data_ptr(), n, o.data_ptr(), scratch.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    want = float((a.double() * b.double()).sum())
    assert abs(float(out[0]) - want) <= 1e-6 * abs(want), (float(out[0]), want)
    assert torch.equal(out[0], out[1])
