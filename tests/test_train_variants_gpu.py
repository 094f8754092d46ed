"""
GPU parity of the loss step for the model variants TimbreTrapFiLM, TimbreTrapMag and TimbreTrapMagDB (reference modules.py:780-1075):
whole-step parameter gradients against the CPU oracle's fp32 autograd (same gates as tests/test_train_gpu.py), the two kernels of their
edges (tt_film_convin_grad, tt_channel0_activation_bwd) against torch autograd, compute_step_losses against the oracle and (for the
base model too) against TrainStep.losses, and a short training run per variant.  The reconstruction target of a variant is its own
encoder input (oracle features_ref).
"""
import contextlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import check_step_gradients, tonal_clip

pytestmark = pytest.mark.gpu

SMALL = dict(sample_rate=8000, n_octaves=6, bins_per_octave=12, secs_per_block=0.5)
BASE = dict(sample_rate=22050, n_octaves=9, bins_per_octave=60, secs_per_block=3)
GEOMETRY = dict(small=SMALL, base=BASE)
CLASSES = dict(base='TimbreTrap', film='TimbreTrapFiLM', mag='TimbreTrapMag', magdb='TimbreTrapMagDB')


def _setup(tag, skip=False, latent=None, complexity=1, geometry='small'):
    """SMALL: two blocks of three clips, two of them with transcription targets; BASE: one 3 s block of one clip."""
    from oracle import model_ref as R
    from timbre_trap_b200 import framework as FW
    geo = GEOMETRY[geometry]
    model = getattr(FW, CLASSES[tag])(latent_size=latent, model_complexity=complexity, skip_connections=skip, **geo)
    sd = R.init_state_dict(model.sliCQ.n_bins, latent, complexity, seed=3, variant=tag)
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


def _oracle_losses(R, tag, sd, c, audio, gt):
    rec, lat, trn, trn_rec, trn_scr = R.forward_variant_ref(tag, audio, sd, c, consistency=True)
    act = R.activations_variant_ref(tag, trn)
    losses = dict(reconstruction=R.reconstruction_loss_ref(rec, R.features_ref(tag, audio, c)),
                  transcription=R.transcription_loss_ref(act[:gt.size(0)], gt, True))
    n = gt.size(0)                                  # the first n clips have transcription targets
    losses['consistency_spectral'], losses['consistency_score'] = R.consistency_loss_ref(trn_rec[:n], trn_scr[:n], trn[:n])
    return losses


@contextlib.contextmanager
def _oracle_relu_decisions(masks):
    """The oracle's ReLU heads (decode_variant_ref of 'mag', called for rec, trn, trn_rec, trn_scr in that order) with the on/off
    decisions of the product's forward.  A ReLU's derivative jumps at 0, so decoder outputs within the bf16 forward's noise of 0
    (about 1e-2 of their scale) take the other branch in one of the two: that alone moves the fp32 oracle's global gradient by
    1.5e-2 - 4.7e-2 rel-L2 (mask flipped by Gaussian noise of 0.3 - 2 % of the rms).  With the same decisions the comparison
    measures the kernels, not the discontinuity."""
    it = iter(masks)
    relu = F.relu
    torch.nn.functional.relu = lambda x, inplace=False: x * next(it).to(x.dtype)
    try:
        yield
    finally:
        torch.nn.functional.relu = relu


def _oracle_grads(R, tag, sd, c, audio, gt):
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    total = sum(_oracle_losses(R, tag, sd, c, audio, gt).values())
    total.backward()
    return {k: v.grad for k, v in sd.items()}, float(total.detach())


def _global_err(got, want):
    num = sum(float((got[k] - want[k]).norm()) ** 2 for k in want)
    return (num / sum(float(v.norm()) ** 2 for v in want.values())) ** 0.5


# film: latent 24 is padded to 32 in the kernels; latent 200 to 256, the latent weight gradients in two slices of 128 channels
CASES = [('film', True, 24), ('film', False, 200), ('mag', False, None), ('magdb', True, None)]


# model_complexity 2 (SMALL geometry): FiLM at latent 128, and MagDB with skips
STEP_CASES = [pytest.param(*case, 1, 'small', id='-'.join(map(str, case))) for case in CASES] + [
    pytest.param('film', False, 128, 2, 'small', id='film-False-128-complexity2-small'),
    pytest.param('magdb', True, None, 2, 'small', id='magdb-True-None-complexity2-small')]
FLOORLESS = 4e-2       # per-parameter rel-L2 without the floor, complexity 2 (measured on a B200: 2.1e-2 FiLM, 1.1e-2 MagDB)


@pytest.mark.parametrize('tag,skip,latent,complexity,geometry', STEP_CASES)
def test_variant_step_gradients_match_oracle_autograd(tag, skip, latent, complexity, geometry):
    from timbre_trap_b200.framework.train import TrainStep
    R, model, sd, c, audio, gt = _setup(tag, skip, latent, complexity, geometry)
    want, want_total = _oracle_grads(R, tag, sd, c, audio, gt)
    masks = None
    if tag == 'mag':
        with torch.no_grad():
            out = model(audio.cuda(), consistency=True)
        masks = [(out[i] > 0).cpu() for i in (0, 2, 3, 4)]
    ts = TrainStep(model)
    out = ts.losses(audio.cuda(), gt.cuda())
    np.testing.assert_allclose(float(out['total'].detach()), want_total, rtol=3e-2)
    ts.backward(out['total'])
    got = {k: p.grad.detach().cpu() for k, p in model.named_parameters()}
    if masks is not None:
        print(f'{tag}: global gradient rel-L2 error against the plain oracle', _global_err(got, want))
        with _oracle_relu_decisions(masks):
            want, _ = _oracle_grads(R, tag, sd, c, audio, gt)
    if tag == 'film':
        assert {'film_layer.gamma.weight', 'film_layer.gamma.bias', 'film_layer.beta.weight', 'film_layer.beta.bias'} <= set(got)
    check_step_gradients(got, want, f'{tag} skip={skip} latent={latent} complexity={complexity} {geometry}',
                         floorless=FLOORLESS if complexity == 2 else None)


def _film_operands(D, C0, H, T, B, seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn((B, D, T), generator=g).to(torch.bfloat16).float()
    dz = (torch.randn((B, C0, H, T), generator=g) * 0.1).to(torch.bfloat16).float()
    w = torch.randn((D, C0, H, 1), generator=g) * 0.1
    film = [torch.randn(s, generator=g) for s in ((D, 2), (D,), (D, 2), (D,))]
    return z, dz, w, film


@pytest.mark.parametrize('D,C0,H,T,B', [(24, 32, 2, 256, 3), (200, 64, 31, 128, 2)])
@pytest.mark.parametrize('hot', [0, 1])
def test_film_convin_gradients_match_autograd(D, C0, H, T, B, hot):
    """tt_film_convin_grad (after the tensor-core sums of tt_conv_wgrad_lat) and the latent gradient against torch autograd of
    conv_transpose2d(film(z)) on the same bf16-rounded z and output gradient, for both conditions.  The weight / bias / Linear gradients
    are fp32 (gate 2e-4 max, as the weight-gradient kernels); the latent gradient is a bf16 tensor computed from the bf16-rounded W * gamma,
    so its reference uses that rounded weight and its gate adds one bf16 rounding of the result (2^-8 relative)."""
    from timbre_trap_b200.framework import layer_grads as LG, packing as P
    from timbre_trap_b200.framework.modules import _latent_pad
    z, dz, w, film = _film_operands(D, C0, H, T, B, seed=D + hot)
    cond = torch.tensor([1.0 - hot, float(hot)])                        # one-hot [transcribe, not transcribe]
    wt, bt = w.clone().requires_grad_(True), torch.zeros(C0, requires_grad=True)
    ft = [f.clone().requires_grad_(True) for f in film]
    zt = z.clone().requires_grad_(True)
    gamma, beta = F.linear(cond, ft[0], ft[1]), F.linear(cond, ft[2], ft[3])
    u = zt * gamma.view(1, -1, 1) + beta.view(1, -1, 1)
    (F.conv_transpose2d(u.unsqueeze(2), wt, bt) * dz).sum().backward()

    d_pad = _latent_pad(D)
    lat8 = P.to_c8(F.pad(z, (0, 0, 0, d_pad - D)).unsqueeze(2).cuda())
    dz8 = P.to_c8(dz.cuda())
    P._PackedCache.epoch += 1                                           # fresh backward packs for these tensors
    args = (dz8, lat8, w.cuda(), *[f.cuda() for f in film], hot, D, C0)
    first = LG._film_convin_grads(*args)
    again = LG._film_convin_grads(*args)
    assert all(torch.equal(a, b) for a, b in zip(first, again))        # fixed reduction order: bit-reproducible
    glat, dw, db, dgw, dgb, dbw, dbb = first
    for name, got, want in (('dW', dw, wt.grad), ('db', db, bt.grad), ('gamma.weight', dgw, ft[0].grad), ('gamma.bias', dgb, ft[1].grad),
                            ('beta.weight', dbw, ft[2].grad), ('beta.bias', dbb, ft[3].grad)):
        assert got.shape == want.shape, name
        err = float((got.cpu() - want).abs().max())
        assert err <= 2e-4 * float(want.abs().max()) + 1e-4, (name, err, float(want.abs().max()))
    assert float(dgw[:, 1 - hot].abs().max()) == 0.0 and float(dbw[:, 1 - hot].abs().max()) == 0.0
    # latent gradient: dz contracted with W * gamma over (c, h), the product's operand rounded to bf16 like the packed weights
    wg = (w * gamma.detach().view(-1, 1, 1, 1)).to(torch.bfloat16).double()[..., 0]
    want_lat = torch.einsum('dch,bcht->bdt', wg, dz.double()).float()
    got_lat = P.from_c8(glat, D)[:, :, 0].cpu()
    err = (got_lat - want_lat).abs()
    assert bool((err <= 2 ** -8 * want_lat.abs() + 2e-4 * float(want_lat.abs().max())).all()), float(err.max())
    # and the same against autograd's fp32 latent gradient, within the bf16 rounding of W * gamma
    assert float((got_lat - zt.grad).abs().max()) <= 1e-2 * float(zt.grad.abs().max())


@pytest.mark.parametrize('mode', [0, 1, 2, 3])
def test_channel0_activation_bwd_matches_autograd(mode):
    from timbre_trap_b200 import _lib
    from timbre_trap_b200.framework import layer_grads as LG
    g = torch.Generator().manual_seed(mode)
    pairs = torch.randn((2, 37, 129, 2), generator=g)
    pairs[0, :5, :, 0] = 0.0                                            # exact zeros: relu'(0) = 0
    gout = torch.randn((2, 37, 129, 2), generator=g)
    v = pairs[..., 0].clone().requires_grad_(True)
    f = {0: lambda x: x, 1: torch.relu, 2: torch.sigmoid, 3: lambda x: torch.tanh(torch.relu(x))}[mode]
    (f(v) * gout[..., 0]).sum().backward()
    got = LG._channel0_bwd(pairs.cuda(), gout.cuda(), mode).cpu()
    assert torch.equal(got[..., 1], torch.zeros_like(got[..., 1]))
    np.testing.assert_allclose(got[..., 0].numpy(), v.grad.numpy(), rtol=1e-5, atol=1e-6)
    with pytest.raises(_lib.TimbreTrapB200Error):
        LG._channel0_bwd(pairs.cuda(), gout.cuda(), 4)


@pytest.mark.parametrize('tag,skip,latent', CASES)
def test_variant_step_losses_match_oracle(tag, skip, latent):
    from timbre_trap_b200.framework.train import compute_step_losses
    R, model, sd, c, audio, gt = _setup(tag, skip, latent)
    got = compute_step_losses(model.eval(), audio.cuda(), gt.cuda())
    with torch.no_grad():
        want = _oracle_losses(R, tag, sd, c, audio, gt)
        trn = R.forward_variant_ref(tag, audio, sd, c)[2]
    want['total'] = sum(want.values())
    # as in tests/test_train_losses_gpu.py: besides the relative tolerance an absolute floor of (bf16 noise level)^2 x the energy of
    # the compared tensors, where the consistency terms of a random-init model sit (the two decodes of one latent are almost identical)
    energy = float(R.reconstruction_loss_ref(trn[:2], torch.zeros_like(trn[:2])))
    for k, v in want.items():
        print(tag, k, float(got[k]), float(v))
        np.testing.assert_allclose(float(got[k]), float(v), rtol=3e-2, atol=(1.5e-2) ** 2 * energy, err_msg=k)


@pytest.mark.parametrize('tag,skip,latent', [('base', False, None), ('base', True, None), ('film', True, 24), ('mag', False, None),
                                             ('magdb', True, None)])
def test_step_losses_equal_train_step_losses(tag, skip, latent):
    """compute_step_losses runs the model's inference layers, TrainStep.losses the same layers through their autograd Functions: the
    same kernels in the same order (the residual blocks' tt_res_block_rs_mid only stores the inner tile tt_res_block_rs stages), so
    every loss agrees bit for bit."""
    from timbre_trap_b200.framework.train import TrainStep, compute_step_losses
    R, model, sd, c, audio, gt = _setup(tag, skip, latent)
    want = compute_step_losses(model, audio.cuda(), gt.cuda())
    got = {k: v.detach() for k, v in TrainStep(model).losses(audio.cuda(), gt.cuda()).items()}
    assert list(got) == list(want)
    for k in want:
        assert torch.equal(got[k], want[k]), (k, float(got[k]), float(want[k]))


def _oracle_training(R, tag, sd, c, audio, gt, steps, lr):
    """Totals of `steps` fp32 oracle steps with torch's clip_grad_norm_(10) + AdamW (train.py:493-496)."""
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.AdamW(list(sd.values()), lr=lr)
    totals = []
    for _ in range(steps):
        total = sum(_oracle_losses(R, tag, sd, c, audio, gt).values())
        opt.zero_grad()
        total.backward()
        torch.nn.utils.clip_grad_norm_(list(sd.values()), 10.0)
        opt.step()
        totals.append(float(total.detach()))
    return totals


# the fp32 oracle's own reduction over these 8 steps: film 0.25, mag 0.77, magdb 0.85 - the decibel variant's sigmoid head learns
# more slowly, so its bound is the oracle's ratio with a margin instead of the base model's 0.8
REDUCTION = dict(film=0.8, mag=0.8, magdb=0.9)


@pytest.mark.parametrize('tag,skip,latent', [('film', False, 24), ('mag', False, None), ('magdb', False, None)])
def test_variant_training_reduces_the_loss(tag, skip, latent):
    from timbre_trap_b200.framework.train import TrainStep
    R, model, sd, c, audio, gt = _setup(tag, skip, latent)
    ts = TrainStep(model, lr=2e-3)
    first = float(ts.step(audio.cuda(), gt.cuda())['total'])
    for _ in range(7):
        last = ts.step(audio.cuda(), gt.cuda())
    want = _oracle_training(R, tag, sd, c, audio, gt, 8, 2e-3)
    print(tag, 'first / last total', first, float(last['total']), 'oracle', want[0], want[-1])
    assert float(last['total']) < REDUCTION[tag] * first, (first, float(last['total']))
    np.testing.assert_allclose(float(last['total']), want[-1], rtol=3e-2)         # the same trajectory as the fp32 oracle
    assert np.isfinite(float(last['grad_norm']))
