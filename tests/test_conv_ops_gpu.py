"""
GPU parity of every conv entry point of the C ABI against torch fp32 convs of the same bf16-rounded inputs and
weights (the kernels compute bf16 x bf16 -> fp32 and round activations to bf16 between layers; tolerance is the
bf16 output rounding, 2^-8 relative, plus fp32 accumulation noise).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rand(shape, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale)


def _bf(x):
    return x.to(torch.bfloat16).float()


@pytest.fixture
def force_strip_rows():
    """tt_set_strip_rows(rows) for the duration of one test (automatic split restored afterwards)."""
    from timbre_trap_b200 import _lib
    yield lambda rows: _lib.check(_lib.lib().tt_set_strip_rows(rows))
    _lib.lib().tt_set_strip_rows(0)


def _rows(rows, linear):
    """Parameter rows of a conv with its ELU epilogue (act=True, ids as they were) and `linear` rows of the same conv without it
    (act=False: the linear epilogue the backward pass runs its data gradients through)."""
    return ([pytest.param(*r, True, id='-'.join(map(str, r))) for r in rows] +
            [pytest.param(*r, False, id='-'.join(map(str, r)) + '-linear') for r in linear])


def _assert_close(got, want, tol=1.2e-2):
    err = float((got - want).abs().max())
    ref = float(want.abs().max())
    assert err <= tol * ref, (err, ref)


@pytest.mark.parametrize('Cin,Cout,H,T,B,act', _rows([(4, 8, 540, 128, 1), (8, 16, 269, 256, 2), (16, 32, 133, 128, 1), (32, 64, 65, 256, 2),
                                                    (2, 4, 20, 100, 1), (8, 16, 7, 128, 1)],
                                                   [(32, 64, 65, 1024, 1), (16, 32, 133, 256, 2), (8, 16, 269, 128, 1), (4, 8, 540, 1024, 1)]))
@pytest.mark.parametrize('strip_rows', [None, 5])
def test_conv_down_strip(Cin, Cout, H, T, B, act, strip_rows, force_strip_rows):
    from timbre_trap_b200.framework import ops, packing as P
    if strip_rows:
        force_strip_rows(strip_rows)
    x = _bf(_rand((B, Cin, H, T), 11))
    w, b = _bf(_rand((Cout, Cin, 4, 1), 12, 0.3)), _rand((Cout,), 13, 0.3)
    want = F.conv2d(x, w, b, stride=(2, 1))
    want = F.elu(want) if act else want
    y = ops.conv_down_strip(P.to_c8(x.cuda()), P.pack_down_strip(w.cuda(), b.cuda()), P.pad8(Cout), act=act)
    assert y.shape[2] == want.shape[2]
    _assert_close(P.from_c8(y, Cout).cpu(), want)


@pytest.mark.parametrize('Cin,Cout,H,T,B', [(4, 8, 540, 256, 1), (2, 4, 20, 100, 2), (3, 7, 31, 516, 1)])
def test_conv_down_packed4_input(Cin, Cout, H, T, B):
    from timbre_trap_b200.framework import ops, packing as P
    x = _bf(_rand((B, Cin, H, T), 11))
    w, b = _bf(_rand((Cout, Cin, 4, 1), 12, 0.3)), _rand((Cout,), 13, 0.3)
    want = F.elu(F.conv2d(x, w, b, stride=(2, 1)))
    y = ops.conv_down_strip(P.to_p4(x.cuda()), P.pack_down_pairs(w.cuda(), b.cuda()), 8)
    assert y.shape == (B, 1, want.shape[2], T, 8)
    _assert_close(P.from_c8(y, Cout).cpu(), want)


@pytest.mark.parametrize('Cin,Cout,H,T,op,B', [(8, 4, 269, 256, 0, 1), (4, 2, 9, 100, 1, 2), (8, 3, 17, 128, 1, 1)])
def test_conv_up_packed4_output(Cin, Cout, H, T, op, B):
    from timbre_trap_b200.framework import ops, packing as P
    x = _bf(_rand((B, Cin, H, T), 21))
    w, b = _bf(_rand((Cin, Cout, 4, 1), 22, 0.3)), _rand((Cout,), 23, 0.3)
    want = F.elu(F.conv_transpose2d(x, w, b, stride=(2, 1), output_padding=(op, 0)))
    y = ops.conv_up_strip(P.to_c8(x.cuda()), P.pack_up_strip(w.cuda(), b.cuda()), 8, op, packed4_out=True)
    assert y.shape == (B, want.shape[2], T, 4)
    _assert_close(P.from_p4(y, Cout).cpu(), want)
    if Cout < 4:
        assert float(y[..., Cout:].float().abs().max()) == 0.0


def test_conv_in_out_packed4():
    from timbre_trap_b200.framework import ops, packing as P
    B, C0, H, T = 2, 4, 33, 260
    x = _rand((B, 2, H, T), 41)
    w, b = _rand((C0, 2, 3, 3), 42, 0.4), _rand((C0,), 43, 0.3)
    want = F.elu(F.conv2d(x, w, b, padding=1))
    y = ops.conv_in(x.permute(0, 2, 3, 1).contiguous().cuda(), w.cuda().contiguous(), b.cuda(), C0, packed4=True)
    assert y.shape == (B, H, T, 4)
    _assert_close(P.from_p4(y, C0).cpu(), want)
    xo = _bf(_rand((B, C0, H, T), 44))
    wo, bo = _rand((2, C0, 3, 3), 45, 0.4), _rand((2,), 46, 0.3)
    yo = ops.conv_out(P.to_p4(xo.cuda()), wo.cuda().contiguous(), bo.cuda(), C0)
    _assert_close(yo.permute(0, 3, 1, 2).cpu(), F.conv2d(xo, wo, bo, padding=1), tol=1e-5)


@pytest.mark.parametrize('Cin,Cout,H,T,op,B,act', _rows([(64, 32, 31, 128, 1, 2), (32, 16, 65, 256, 1, 1), (16, 8, 133, 128, 1, 2),
                                                       (8, 4, 269, 256, 0, 1), (4, 2, 9, 100, 1, 1), (16, 8, 5, 128, 0, 1)],
                                                      [(8, 4, 269, 1024, 0, 1), (16, 8, 133, 256, 1, 2), (32, 16, 65, 1024, 1, 1),
                                                       (64, 32, 31, 128, 1, 2)]))
@pytest.mark.parametrize('strip_rows', [None, 3])
def test_conv_up_strip(Cin, Cout, H, T, op, B, act, strip_rows, force_strip_rows):
    from timbre_trap_b200.framework import ops, packing as P
    if strip_rows:
        force_strip_rows(strip_rows)
    x = _bf(_rand((B, Cin, H, T), 21))
    w, b = _bf(_rand((Cin, Cout, 4, 1), 22, 0.3)), _rand((Cout,), 23, 0.3)
    want = F.conv_transpose2d(x, w, b, stride=(2, 1), output_padding=(op, 0))
    want = F.elu(want) if act else want
    y = ops.conv_up_strip(P.to_c8(x.cuda()), P.pack_up_strip(w.cuda(), b.cuda()), P.pad8(Cout), op, act=act)
    assert y.shape[2] == want.shape[2]
    _assert_close(P.from_c8(y, Cout).cpu(), want)


@pytest.mark.parametrize('C4,H4,D,T,B,act', _rows([(64, 31, 128, 256, 2), (32, 2, 32, 128, 1), (64, 2, 24, 100, 2), (64, 31, 240, 256, 1)],
                                                  [(64, 31, 128, 1024, 1), (32, 31, 32, 256, 2), (64, 2, 24, 100, 2)]))
def test_conv_lat_and_deconv_in(C4, H4, D, T, B, act):
    """act=False: deconv_in's linear epilogue, the data gradient of Encoder.convlat in the loss step."""
    from timbre_trap_b200.framework import ops, packing as P
    from timbre_trap_b200.framework.modules import _latent_pad
    Dp = _latent_pad(D)
    x = _bf(_rand((B, C4, H4, T), 31))
    w, b = _bf(_rand((D, C4, H4, 1), 32, 0.05)), _rand((D,), 33, 0.3)
    want = F.conv2d(x, w, b)
    lat = ops.conv_lat(P.to_c8(x.cuda()), P.pack_lat(w.cuda(), Dp), P.pad_vec(b.cuda(), Dp), Dp)
    _assert_close(P.from_c8(lat, D).cpu(), want)
    if Dp > D:                                                          # padded latent channels: zero weights, zero bias
        assert float(lat.float().permute(0, 1, 4, 2, 3).reshape(B, Dp, T)[:, D:].abs().max()) == 0.0
    # decoder side
    wd, bd = _bf(_rand((D + 1, C4, H4, 1), 34, 0.1)), _rand((C4,), 35, 0.3)
    lat_in = _bf(_rand((B, D, 1, T), 36))
    packed, tables = P.pack_deconv_in(wd.cuda(), bd.cuda(), Dp)
    for mode, flag in ((0, 0.0), (1, 1.0)):
        full = torch.cat((lat_in, torch.full((B, 1, 1, T), flag)), dim=1)
        wantd = F.conv_transpose2d(full, wd, bd)
        wantd = F.elu(wantd) if act else wantd
        y = ops.deconv_in(P.to_c8(lat_in.cuda()) if Dp == P.pad8(D) else P.to_c8(F.pad(lat_in, (0, 0, 0, 0, 0, Dp - D)).cuda()),
                          packed, tables[mode].contiguous(), P.pad8(C4), H4, act=act)
        _assert_close(P.from_c8(y, C4).cpu(), wantd)


@pytest.mark.parametrize('C0,H,T,B,packed4', [pytest.param(*r, 0, id='-'.join(map(str, r)))
                                               for r in [(4, 60, 300, 2), (2, 33, 128, 1), (8, 17, 64, 1), (4, 5, 1024, 1), (3, 9, 516, 2)]] +
                                              [pytest.param(*r, 2, id='-'.join(map(str, r)) + '-packed-linear')
                                               for r in [(4, 540, 1024, 1), (2, 72, 200, 2), (3, 9, 516, 2)]])
def test_conv_in_out(C0, H, T, B, packed4):
    """packed4=2: packed 4-channel output without the ELU, the data gradient of Decoder.convout in the loss step."""
    from timbre_trap_b200.framework import ops, packing as P
    x = _rand((B, 2, H, T), 41)
    w, b = _rand((C0, 2, 3, 3), 42, 0.4), _rand((C0,), 43, 0.3)
    want = F.conv2d(x, w, b, padding=1)
    y = ops.conv_in(x.permute(0, 2, 3, 1).contiguous().cuda(), w.cuda().contiguous(), b.cuda(), C0, packed4=packed4)
    if packed4:
        assert y.shape == (B, H, T, 4)
        _assert_close(P.from_p4(y, C0).cpu(), want)
        if C0 < 4:
            assert float(y[..., C0:].float().abs().max()) == 0.0
    else:
        _assert_close(P.from_c8(y, C0).cpu(), F.elu(want))
    xo = _bf(_rand((B, C0, H, T), 44))
    wo, bo = _rand((2, C0, 3, 3), 45, 0.4), _rand((2,), 46, 0.3)
    wanto = F.conv2d(xo, wo, bo, padding=1)
    yo = ops.conv_out(P.to_c8(xo.cuda()), wo.cuda().contiguous(), bo.cuda(), C0)
    _assert_close(yo.permute(0, 3, 1, 2).cpu(), wanto, tol=1e-5)


@pytest.mark.parametrize('C,H,T,k,d,act', [(4, 37, 256, 3, 1, True), (8, 30, 128, 3, 2, False), (8, 19, 384, 1, 1, False), (16, 33, 256, 3, 3, True),
                                            (16, 21, 128, 1, 1, True), (32, 65, 256, 3, 2, False), (32, 17, 128, 1, 1, False), (2, 7, 512, 3, 1, False),
                                            (8, 7, 512, 3, 3, False), (4, 16, 512, 1, 1, False)])
def test_conv_same(C, H, T, k, d, act):
    """The single-stage tile-kernel conv used by the backward pass (recompute and data gradients); repeated to catch races."""
    from timbre_trap_b200.framework import ops, packing as P
    B = 3
    x = _bf(_rand((B, C, H, T), 1))
    w = _bf(_rand((C, C, k, k), 2, 0.3))
    b = _rand((C,), 3, 0.3) if act else None
    want = F.conv2d(x, w, b, padding=d if k == 3 else 0, dilation=d if k == 3 else 1)
    want = F.elu(want) if act else want
    n = max(16, P.pad8(C))
    wp = P.pack_res3x3(w.cuda()) if k == 3 else P.pack_res1x1(w.cuda())
    x8 = P.to_c8(x.cuda())
    for _ in range(4):
        y = ops.conv_same(x8, wp, P.pad_vec(b.cuda(), n) if b is not None else None, k, d, act=act)
        _assert_close(P.from_c8(y, C).cpu(), want)


@pytest.mark.parametrize('C,H,T,d,B', [(4, 37, 256, 1, 2), (8, 30, 128, 2, 1), (8, 19, 384, 3, 2), (16, 33, 256, 1, 2),
                                         (16, 21, 128, 3, 1), (32, 65, 256, 2, 1), (32, 17, 128, 3, 2), (2, 20, 200, 1, 1),
                                         (4, 540, 128, 3, 1), (32, 5, 128, 3, 1), (16, 2, 100, 2, 3), (16, 67, 128, 2, 1),
                                         (32, 70, 128, 1, 1)])
@pytest.mark.parametrize('strip_rows', [None, 7, 2])
def test_res_block_rs(C, H, T, d, B, strip_rows, force_strip_rows):
    """Row-stationary residual block (csrc/res_rs.cu): image edges, strip seams (rows per strip below the dilation included),
    TMEM ring wrap-around (H well above the slot count)."""
    from timbre_trap_b200.framework import ops, packing as P
    if strip_rows:
        force_strip_rows(strip_rows)
    x = _bf(_rand((B, C, H, T), 1))
    w1, b1 = _bf(_rand((C, C, 3, 3), 2, 0.3)), _rand((C,), 3, 0.3)
    w2, b2 = _bf(_rand((C, C, 1, 1), 4, 0.5)), _rand((C,), 5, 0.3)
    mid = _bf(F.elu(F.conv2d(x, w1, b1, padding=d, dilation=d)))
    want = x + F.elu(F.conv2d(mid, w2, b2))
    w1p, w2p, bias = P.pack_res_rs(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda())
    y = ops.res_block_rs(P.to_c8(x.cuda()), w1p, w2p, bias, C, d)
    torch.cuda.synchronize()
    _assert_close(P.from_c8(y, C).cpu(), want)
    if P.pad8(C) != C:
        assert float(y.float().permute(0, 1, 4, 2, 3).reshape(B, -1, H, T)[:, C:].abs().max()) == 0.0


@pytest.mark.parametrize('C,H,T,d,B', [(4, 37, 256, 1, 2), (4, 30, 512, 2, 1), (4, 540, 256, 3, 1), (2, 20, 200, 1, 1), (3, 9, 260, 3, 2),
                                         (4, 3, 1024, 2, 1)])
@pytest.mark.parametrize('strip_rows', [None, 7, 1])
def test_res_block_rs_packed4(C, H, T, d, B, strip_rows, force_strip_rows):
    from timbre_trap_b200.framework import ops, packing as P
    if strip_rows:
        force_strip_rows(strip_rows)
    x = _bf(_rand((B, C, H, T), 1))
    w1, b1 = _bf(_rand((C, C, 3, 3), 2, 0.3)), _rand((C,), 3, 0.3)
    w2, b2 = _bf(_rand((C, C, 1, 1), 4, 0.5)), _rand((C,), 5, 0.3)
    mid = _bf(F.elu(F.conv2d(x, w1, b1, padding=d, dilation=d)))
    want = x + F.elu(F.conv2d(mid, w2, b2))
    w1p, w2p, bias = P.pack_res_rs_pairs(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda(), d)
    y = ops.res_block_rs(P.to_p4(x.cuda()), w1p, w2p, bias, 4, d)
    torch.cuda.synchronize()
    _assert_close(P.from_p4(y, C).cpu(), want)
    if C < 4:
        assert float(y[..., C:].float().abs().max()) == 0.0


@pytest.mark.parametrize('C,H,T,d,B,fold', [(4, 37, 512, 1, 2, 4), (4, 30, 1024, 2, 1, 4), (4, 540, 512, 3, 1, 4), (2, 20, 200, 1, 1, 4),
                                              (3, 9, 260, 3, 2, 4), (8, 30, 256, 1, 2, 2), (8, 269, 512, 2, 1, 2), (8, 19, 384, 3, 2, 2),
                                              (5, 12, 130, 3, 1, 2), (8, 3, 1024, 1, 1, 2)])
@pytest.mark.parametrize('strip_rows', [None, 7])
def test_res_block_rs_folded(C, H, T, d, B, fold, strip_rows, force_strip_rows):
    """Folded rows: 4 frames x 4 channels of the packed layout, or 2 frames x 8 channels of C8 planar, per GEMM row."""
    from timbre_trap_b200.framework import ops, packing as P
    if strip_rows:
        force_strip_rows(strip_rows)
    x = _bf(_rand((B, C, H, T), 1))
    w1, b1 = _bf(_rand((C, C, 3, 3), 2, 0.3)), _rand((C,), 3, 0.3)
    w2, b2 = _bf(_rand((C, C, 1, 1), 4, 0.5)), _rand((C,), 5, 0.3)
    mid = _bf(F.elu(F.conv2d(x, w1, b1, padding=d, dilation=d)))
    want = x + F.elu(F.conv2d(mid, w2, b2))
    w1p, w2p, bias = P.pack_res_rs_fold(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda(), d, fold)
    xin = P.to_p4(x.cuda()) if fold == 4 else P.to_c8(x.cuda())
    y = ops.res_block_rs(xin, w1p, w2p, bias, C, d, fold=True)
    torch.cuda.synchronize()
    got = P.from_p4(y, C) if fold == 4 else P.from_c8(y, C)
    _assert_close(got.cpu(), want)
    pad = y[..., C:] if fold == 4 else y.float().permute(0, 1, 4, 2, 3).reshape(B, -1, H, T)[:, C:]
    if pad.numel():
        assert float(pad.float().abs().max()) == 0.0


@pytest.mark.parametrize('C,H,T,d,mode', [(4, 23, 256, 1, 'fold4'), (3, 17, 130, 2, 'pairs'), (8, 19, 256, 3, 'fold2'), (8, 9, 131, 1, 'planar'),
                                          (16, 21, 200, 2, 'planar'), (32, 11, 128, 3, 'planar')])
def test_res_block_inner_activation_output(C, H, T, d, mode):
    """tt_res_block_rs_mid: the block's output is unchanged (bit for bit) and `mid` holds ELU(conv3x3(x) + b1) as the kernel stages it
    for its 1x1 conv (bf16) - what the loss step keeps for its backward pass."""
    import torch.nn.functional as F
    from timbre_trap_b200.framework import ops, packing as P
    g = torch.Generator().manual_seed(C * 10 + d)
    x = torch.randn((2, C, H, T), generator=g)
    w1, b1 = torch.randn((C, C, 3, 3), generator=g) * 0.2, torch.randn(C, generator=g) * 0.1
    w2, b2 = torch.randn((C, C, 1, 1), generator=g) * 0.3, torch.randn(C, generator=g) * 0.1
    packed = mode in ('fold4', 'pairs')
    xin = (P.to_p4(x) if packed else P.to_c8(x)).cuda()
    if mode == 'fold4':
        pk = P.pack_res_rs_fold(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda(), d, 4)
    elif mode == 'fold2':
        pk = P.pack_res_rs_fold(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda(), d, 2)
    elif mode == 'pairs':
        pk = P.pack_res_rs_pairs(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda(), d)
    else:
        pk = P.pack_res_rs(w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda())
    fold = mode.startswith('fold')
    y0 = ops.res_block_rs(xin, *pk, C, d, fold=fold)
    mid = torch.full_like(xin, float('nan'))
    y1 = ops.res_block_rs(xin, *pk, C, d, fold=fold, mid_out=mid)
    assert torch.equal(y0, y1)
    got = (P.from_p4(mid, C) if packed else P.from_c8(mid, C)).cpu()
    xb = x.to(torch.bfloat16).float()
    want = F.elu(F.conv2d(xb, w1.to(torch.bfloat16).float(), b1, padding=d, dilation=d))
    assert torch.isfinite(got).all()
    assert float((got - want).abs().max()) <= 2e-2 * max(1.0, float(want.abs().max()))
    with pytest.raises(ValueError):
        ops.res_block_rs(xin, *pk, C, d, fold=fold, mid_out=mid[:1])


@pytest.mark.parametrize('C,H,T,k,d', [(8, 13, 200, 1, 1), (16, 21, 128, 3, 2), (32, 9, 256, 3, 3), (5, 7, 131, 3, 1)])
def test_conv_same_fused_epilogues(C, H, T, k, d):
    """tt_conv_same_post: the element-wise passes of the residual blocks' backward in the conv's epilogue - times ELU'(.) given the
    activated tensor (the 1x1 data gradient), plus a tensor (the residual add of the 3x3 data gradient)."""
    from timbre_trap_b200.framework import ops, packing as P
    B = 2
    x = _bf(_rand((B, C, H, T), 1))
    w = _bf(_rand((C, C, k, k), 2, 0.3))
    e = _bf(_rand((B, C, H, T), 7))
    conv = F.conv2d(x, w, None, padding=d if k == 3 else 0, dilation=d if k == 3 else 1)
    wp = P.pack_res3x3(w.cuda()) if k == 3 else P.pack_res1x1(w.cuda())
    x8, e8 = P.to_c8(x.cuda()), P.to_c8(e.cuda())
    got = ops.conv_same(x8, wp, None, k, d, times_elu_grad_of=e8)
    _assert_close(P.from_c8(got, C).cpu(), conv * torch.where(e > 0, torch.ones_like(e), e + 1))
    got = ops.conv_same(x8, wp, None, k, d, plus=e8)
    _assert_close(P.from_c8(got, C).cpu(), conv + e)
    with pytest.raises(ValueError):
        ops.conv_same(x8, wp, None, k, d, plus=e8[:1])
