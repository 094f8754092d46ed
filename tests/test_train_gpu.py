"""
GPU parity of the backward half of the loss step (experiments/train.py:470-496): the weight-gradient kernels against torch
autograd, the whole step's parameter gradients against the CPU oracle's autograd (fp32), and clip + AdamW against torch.optim.
Tolerance on gradients: the forward runs in bf16 and activation gradients travel in bf16 between layers (the reference trains
under fp16 autocast), so per-parameter gradients are compared at rel-L2 <= 1e-1 (the small bias vectors are the noisiest) and the global gradient at 3e-2.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import check_step_gradients, tonal_clip

pytestmark = pytest.mark.gpu

SMALL = dict(sample_rate=8000, n_octaves=6, bins_per_octave=12, secs_per_block=0.5)
BASE = dict(sample_rate=22050, n_octaves=9, bins_per_octave=60, secs_per_block=3)     # bench.py's loss step: 540 bins, T = 1024 per block
GEOMETRY = dict(small=SMALL, base=BASE)


def _setup(skip=False, latent=None, complexity=1, geometry='small'):
    """SMALL: two blocks of three clips, two of them with transcription targets; BASE: one 3 s block of one clip."""
    from oracle import model_ref as R
    from timbre_trap_b200.framework import TimbreTrap
    geo = GEOMETRY[geometry]
    model = TimbreTrap(latent_size=latent, model_complexity=complexity, skip_connections=skip, **geo)
    sd = R.init_state_dict(model.sliCQ.n_bins, latent, complexity, seed=3)
    if skip:
        sd['skip_weights'] = torch.tensor([0.9, 1.1, 0.8, 1.2, 0.7])
    model.load_state_dict(sd)
    model = model.cuda()
    c = R.CQTRef(geo['n_octaves'], geo['bins_per_octave'], geo['sample_rate'], geo['secs_per_block'])
    n_blocks, n_batch, n_gt = (1, 1, 1) if geometry == 'base' else (2, 3, 2)
    audio = tonal_clip(n_blocks * c.block_length, geo['sample_rate'], seed=4, n_batch=n_batch)
    rng = np.random.default_rng(2)
    gt = torch.zeros((n_gt, c.n_bins, n_blocks * c.max_window_length))
    for b in range(n_gt):
        for k in rng.integers(5, c.n_bins - 5, size=3):
            gt[b, k, :] = 1.0
            gt[b, k - 1, :] = gt[b, k + 1, :] = 0.6
    return R, model, sd, c, audio, gt


def _oracle_grads(R, sd, c, audio, gt):
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    coeffs = c(audio)
    rec, lat, trn, trn_rec, trn_scr = R.forward_ref(audio, sd, c, consistency=True)
    act = torch.tanh(c.to_magnitude(trn))
    n = gt.size(0)                                  # the first n clips have transcription targets
    losses = dict(reconstruction=R.reconstruction_loss_ref(rec, coeffs), transcription=R.transcription_loss_ref(act[:n], gt, True))
    losses['consistency_spectral'], losses['consistency_score'] = R.consistency_loss_ref(trn_rec[:n], trn_scr[:n], trn[:n])
    total = sum(losses.values())
    total.backward()
    return {k: v.grad for k, v in sd.items()}, losses, float(total.detach())


# 40 latent channels: padded to 64 in the kernels; 200: padded to 256, the latent weight gradients in two slices of 128 channels.
# model_complexity 2 at the BASE geometry with latent 128 is the benchmarked model: every layer that exists only at complexity 2 (the
# 32-channel residual blocks, the 32 -> 64 sconv, the 64 -> 32 tconv, the 64-channel convlat / convin) at the heights that ship.
STEP_CASES = [pytest.param(False, None, 1, 'small', id='False-None'), pytest.param(True, None, 1, 'small', id='True-None'),
              pytest.param(False, 40, 1, 'small', id='False-40'), pytest.param(False, 200, 1, 'small', id='False-200'),
              pytest.param(True, 128, 2, 'base', id='True-128-complexity2-base'), pytest.param(False, None, 2, 'small', id='False-None-complexity2-small')]
FLOORLESS = 2.5e-2       # per-parameter rel-L2 without the floor, complexity 2 (measured on a B200: 1.2e-2 at SMALL, 8.3e-3 at BASE)


@pytest.mark.parametrize('skip,latent,complexity,geometry', STEP_CASES)
def test_step_gradients_match_oracle_autograd(skip, latent, complexity, geometry):
    from timbre_trap_b200.framework.train import TrainStep
    R, model, sd, c, audio, gt = _setup(skip, latent, complexity, geometry)
    want, want_losses, want_total = _oracle_grads(R, sd, c, audio, gt)
    ts = TrainStep(model)
    out = ts.losses(audio.cuda(), gt.cuda())
    np.testing.assert_allclose(float(out['total'].detach()), want_total, rtol=3e-2)
    ts.backward(out['total'])
    got = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    check_step_gradients(got, want, f'skip={skip} latent={latent} complexity={complexity} {geometry}',
                          floorless=FLOORLESS if complexity == 2 else None)


def test_clip_and_adamw_match_torch():
    from timbre_trap_b200.framework.train import TrainStep
    R, model, sd, c, audio, gt = _setup()
    ts = TrainStep(model, lr=1e-3, max_norm=10.0)
    ref_params = [p.detach().clone().requires_grad_(True) for p in model.parameters()]
    opt = torch.optim.AdamW(ref_params, lr=1e-3)
    g = torch.Generator(device='cuda').manual_seed(0)
    for step in range(3):
        for p, q in zip(model.parameters(), ref_params):
            p.grad = torch.randn(p.shape, device='cuda', generator=g) * (30.0 if step == 1 else 0.01)   # step 1 is clipped
            q.grad = p.grad.clone()
        norm = ts.optimizer_step()
        ref_norm = torch.nn.utils.clip_grad_norm_(ref_params, 10.0)
        opt.step()
        assert abs(float(norm) - float(ref_norm)) <= 1e-4 * float(ref_norm)
        for p, q in zip(model.parameters(), ref_params):
            assert torch.allclose(p.detach(), q.detach(), atol=1e-6, rtol=1e-5)


def test_training_reduces_the_loss():
    from timbre_trap_b200.framework.train import TrainStep
    R, model, sd, c, audio, gt = _setup()
    ts = TrainStep(model, lr=2e-3)
    first = float(ts.step(audio.cuda(), gt.cuda())['total'])
    for _ in range(7):
        last = ts.step(audio.cuda(), gt.cuda())
    assert float(last['total']) < 0.8 * first, (first, float(last['total']))
    assert np.isfinite(float(last['grad_norm']))


# the last 16 rows: the residual stages of the BASE geometry at model_complexity 2 (heights 540 / 269 / 133 / 65, T = 1024 frames)
@pytest.mark.parametrize('C,H,T,k,d,B', [(4, 23, 256, 3, 1, 2), (8, 17, 384, 3, 2, 1), (16, 33, 200, 3, 3, 2), (32, 9, 128, 3, 1, 3), (32, 40, 512, 1, 1, 1),
                                           (3, 11, 136, 1, 1, 2), (16, 300, 128, 3, 2, 1), (8, 20, 256, 3, 3, 1), (2, 35, 640, 3, 3, 2)] +
                         [(C, H, 1024, 3, d, 1) for C, H in ((4, 540), (8, 269), (16, 133), (32, 65)) for d in (1, 2, 3)] +
                         [(C, H, 1024, 1, 1, 1) for C, H in ((4, 540), (8, 269), (16, 133), (32, 65))])
def test_tensor_core_weight_gradient(C, H, T, k, d, B):
    """tt_conv_wgrad_same (MN-major tcgen05 GEMM over the pixel axis, deterministic two-stage reduction) against torch autograd on the
    same bf16-rounded operands; products of bf16 values are exact in fp32, so only the summation order differs."""
    import torch.nn.functional as F
    from timbre_trap_b200.framework import layer_grads as LG, packing as P
    g = torch.Generator().manual_seed(C * 100 + H)
    x = torch.randn((B, C, H, T), generator=g).to(torch.bfloat16).float()
    dz = (torch.randn((B, C, H, T), generator=g) * 0.1).to(torch.bfloat16).float()
    w = torch.zeros((C, C, k, k), requires_grad=True)
    bias = torch.zeros(C, requires_grad=True)
    pad = d if k == 3 else 0
    y = F.conv2d(x, w, bias, padding=pad, dilation=d if k == 3 else 1)
    (y * dz).sum().backward()
    dw, db = LG._wgrad_same(P.to_c8(x.cuda()), P.to_c8(dz.cuda()), C, C, k, d)
    assert dw.shape == w.grad.shape
    scale = float(w.grad.abs().max())
    assert float((dw.cpu() - w.grad).abs().max()) <= 2e-4 * scale + 1e-4, (float((dw.cpu() - w.grad).abs().max()), scale)
    assert float((db.cpu() - bias.grad).abs().max()) <= 2e-4 * float(bias.grad.abs().max()) + 1e-4
    dw2, db2 = LG._wgrad_same(P.to_c8(x.cuda()), P.to_c8(dz.cuda()), C, C, k, d)
    assert torch.equal(dw, dw2) and torch.equal(db, db2)                  # fixed reduction order: bit-reproducible


@pytest.mark.parametrize('Cf,Cc,Hc,T,op,B', [(4, 8, 19, 256, 0, 2), (8, 16, 33, 200, 1, 1), (16, 32, 9, 384, 0, 2), (32, 64, 31, 128, 1, 2),
                                             (4, 8, 269, 1024, 0, 1), (8, 16, 133, 1024, 1, 1), (16, 32, 65, 1024, 1, 1)])   # BASE stages
def test_tensor_core_weight_gradient_strided_and_transposed(Cf, Cc, Hc, T, op, B):
    """tt_conv_wgrad_updown against torch autograd: EncoderBlock.sconv (fine = input, coarse = output gradient) and DecoderBlock.tconv
    (coarse = input, fine = output gradient, bias gradient = pixel sums of the fine tensor)."""
    from timbre_trap_b200.framework import layer_grads as LG, packing as P
    g = torch.Generator().manual_seed(Cf * 10 + Hc)
    Hf = 2 * Hc + 2 + op
    fine = torch.randn((B, Cf, Hf, T), generator=g).to(torch.bfloat16).float()
    coarse = (torch.randn((B, Cc, Hc, T), generator=g) * 0.1).to(torch.bfloat16).float()
    # strided conv: y = conv(fine, w (Cc, Cf, 4, 1), stride 2) has (Hf - 4) // 2 + 1 = Hc rows; coarse plays dL/dy
    w = torch.zeros((Cc, Cf, 4, 1), requires_grad=True)
    bias = torch.zeros(Cc, requires_grad=True)
    y = F.conv2d(fine, w, bias, stride=(2, 1))
    assert y.shape[2] == Hc
    (y * coarse).sum().backward()
    dw, db = LG._wgrad_updown(P.to_c8(fine.cuda()), P.to_c8(coarse.cuda()), Cf, Cc, False)
    assert float((dw.cpu() - w.grad).abs().max()) <= 2e-4 * float(w.grad.abs().max()) + 1e-4
    assert float((db.cpu() - bias.grad).abs().max()) <= 2e-4 * float(bias.grad.abs().max()) + 1e-4
    # transposed conv: y = convT(coarse, wt (Cc, Cf, 4, 1), stride 2, output_padding op) has Hf rows; fine plays dL/dy
    wt = torch.zeros((Cc, Cf, 4, 1), requires_grad=True)
    bt = torch.zeros(Cf, requires_grad=True)
    yt = F.conv_transpose2d(coarse, wt, bt, stride=(2, 1), output_padding=(op, 0))
    assert yt.shape[2] == Hf
    (yt * fine).sum().backward()
    dwt, dbt = LG._wgrad_updown(P.to_c8(fine.cuda()), P.to_c8(coarse.cuda()), Cf, Cc, True)
    assert float((dwt.cpu() - wt.grad).abs().max()) <= 2e-4 * float(wt.grad.abs().max()) + 1e-4
    assert float((dbt.cpu() - bt.grad).abs().max()) <= 2e-4 * float(bt.grad.abs().max()) + 2e-3


@pytest.mark.parametrize('Ct,Cf,H,T,B', [(64, 128, 31, 256, 2), (32, 32, 5, 200, 3), (64, 100, 31, 128, 1), (64, 200, 31, 128, 1)])
def test_tensor_core_weight_gradient_tall_kernel_layers(Ct, Cf, H, T, B):
    """tt_conv_wgrad_lat against torch autograd: Encoder.convlat (Conv2d (Cf, Ct, H, 1) over the full height) and Decoder.convin
    (ConvTranspose2d (Cf + 1, Ct, H, 1) with the indicator channel: its weight row and the bias are row sums of the output gradient)."""
    from timbre_trap_b200.framework import layer_grads as LG, packing as P
    g = torch.Generator().manual_seed(Ct + H)
    tall = torch.randn((B, Ct, H, T), generator=g).to(torch.bfloat16).float()
    flat = (torch.randn((B, Cf, 1, T), generator=g) * 0.1).to(torch.bfloat16).float()
    fpad = (Cf + 15) // 16 * 16
    flat8 = P.to_c8(torch.nn.functional.pad(flat, (0, 0, 0, 0, 0, fpad - Cf)).cuda())
    tall8 = P.to_c8(tall.cuda())
    # convlat: y = conv(tall, w (Cf, Ct, H, 1)); flat plays dL/dy
    w = torch.zeros((Cf, Ct, H, 1), requires_grad=True)
    bias = torch.zeros(Cf, requires_grad=True)
    (F.conv2d(tall, w, bias) * flat).sum().backward()
    dw = torch.zeros((Cf, Ct, H, 1), device='cuda')
    db = torch.zeros(Cf, device='cuda')
    LG._wgrad_lat(tall8, flat8, Ct, Cf, dw, db, None)
    assert float((dw.cpu() - w.grad).abs().max()) <= 2e-4 * float(w.grad.abs().max()) + 1e-4
    assert float((db.cpu() - bias.grad).abs().max()) <= 2e-4 * float(bias.grad.abs().max()) + 1e-4
    # decoder convin: y = convT(cat(flat, indicator), wt (Cf + 1, Ct, H, 1)); tall plays dL/dy
    wt = torch.zeros((Cf + 1, Ct, H, 1), requires_grad=True)
    bt = torch.zeros(Ct, requires_grad=True)
    full = torch.cat((flat, torch.ones_like(flat[:, :1])), dim=1)
    (F.conv_transpose2d(full, wt, bt) * tall).sum().backward()
    dwt = torch.zeros((Cf + 1, Ct, H, 1), device='cuda')
    rows = torch.zeros((Ct, H), device='cuda')
    LG._wgrad_lat(tall8, flat8, Ct, Cf, dwt, None, rows)
    dwt[Cf, :, :, 0] = rows
    assert float((dwt.cpu() - wt.grad).abs().max()) <= 2e-4 * float(wt.grad.abs().max()) + 2e-3
    assert float((rows.sum(1).cpu() - bt.grad).abs().max()) <= 2e-4 * float(bt.grad.abs().max()) + 2e-3
