"""
Training through the reference's class API (experiments/train.py:393-500, SURVEY.md section 3.3): `model.train()`,
`model(audio, consistency=True)`, `to_activations`, the three `compute_*_loss` functions, `backward()` - with torch's own optimizer and
clipping.  The step's losses against compute_step_losses, its gradients against the fp32 oracle's autograd and against TrainStep, the
inference path left as it was, frozen parameters, gradients to decode's inputs, the activation and objective gradients, autocast, a
short training run and the bounded backward-pack cache.
"""
import numpy as np
import pytest
import torch

from tests.test_train_variants_gpu import _global_err, _oracle_grads, _oracle_relu_decisions, _setup

pytestmark = pytest.mark.gpu

CASES = [('base', False, None), ('base', True, None), ('film', True, 24), ('film', False, 200), ('mag', False, None), ('magdb', True, None)]


def _launches():
    from timbre_trap_b200 import _lib
    torch.cuda.synchronize()
    return int(_lib.lib().tt_launch_count(1))


def _target(model, tag, audio):
    """The reconstruction target: model.sliCQ(audio) (train.py:404); for the magnitude variants their own one-channel encoder input
    (what TrainStep compares their one-channel output with)."""
    coefficients = model.sliCQ(audio)
    if tag in ('base', 'film'):
        return coefficients
    mag = model.sliCQ.to_magnitude(coefficients)
    return (model.sliCQ.to_decibels(mag) if tag == 'magdb' else mag).unsqueeze(1)


def _reference_step(model, tag, audio, gt):
    """The reference's loop body up to backward() (train.py:404-472) on the public API; returns the losses with their graph."""
    from timbre_trap_b200.framework import compute_consistency_loss, compute_reconstruction_loss, compute_transcription_loss
    model.train()
    coefficients = _target(model, tag, audio)
    rec, _, trn, trn_rec, trn_scr, _ = model(audio, consistency=1)
    act = model.to_activations(trn)
    n = gt.size(0)
    out = dict(reconstruction=compute_reconstruction_loss(rec, coefficients), transcription=compute_transcription_loss(act[:n], gt, True))
    out['consistency_spectral'], out['consistency_score'] = compute_consistency_loss(trn_rec[:n], trn_scr[:n], trn[:n])
    out['total'] = out['reconstruction'] + out['transcription'] + (out['consistency_spectral'] + out['consistency_score'])
    return out


def _grads(model):
    return {k: p.grad.detach().clone().cpu() for k, p in model.named_parameters() if p.grad is not None}


@pytest.mark.parametrize('tag,skip,latent', CASES)
def test_reference_step_losses_and_gradients(tag, skip, latent):
    """The losses equal compute_step_losses (bit for bit where both sum the same elements: the magnitude variants' one-channel
    reconstruction / consistency losses sum (B, 1, F, T) tensors, the loss step their (h, 0) pairs - the same terms in another order),
    the gradients meet the oracle gates of the variant tests and agree with TrainStep's."""
    from timbre_trap_b200.framework.train import TrainStep, compute_step_losses
    R, model, sd, c, audio, gt = _setup(tag, skip, latent)
    audio, gt_d = audio.cuda(), gt.cuda()
    want_losses = compute_step_losses(model, audio, gt_d)
    masks = None
    if tag == 'mag':
        with torch.no_grad():
            o = model.eval()(audio, consistency=True)
        masks = [(o[i] > 0).cpu() for i in (0, 2, 3, 4)]
    out = _reference_step(model, tag, audio, gt_d)
    assert all(v.grad_fn is not None for v in out.values())
    for k in want_losses:
        if tag in ('mag', 'magdb') and k != 'transcription':
            np.testing.assert_allclose(float(out[k].detach()), float(want_losses[k]), rtol=1e-6, err_msg=k)
        else:
            assert torch.equal(out[k].detach(), want_losses[k]), (k, float(out[k]), float(want_losses[k]))
    out['total'].backward()
    got = _grads(model)
    # against the fp32 oracle's autograd (the Mag head's ReLU with the product's on / off decisions, as in the variant tests)
    if masks is not None:
        with _oracle_relu_decisions(masks):
            want, _ = _oracle_grads(R, tag, sd, c, audio.cpu(), gt)
    else:
        want, _ = _oracle_grads(R, tag, sd, c, audio.cpu(), gt)
    assert set(got) == set(want)
    total_norm = sum(float(v.norm()) ** 2 for v in want.values()) ** 0.5
    for k in want:
        err, ref = float((got[k] - want[k]).norm()), float(want[k].norm())
        assert err <= 1e-1 * ref + 1e-2 * total_norm, (k, err, ref, total_norm)
    e_oracle = _global_err(got, want)
    assert e_oracle <= 3e-2, e_oracle
    # against TrainStep on the same model (the transcription's three gradient contributions may add up in another order)
    for p in model.parameters():
        p.grad = None
    ts = TrainStep(model)
    ts.backward(ts.losses(audio, gt_d)['total'])
    e_ts = _global_err(got, _grads(model))
    print(f'{tag} skip={skip} latent={latent}: gradient rel-L2 vs oracle {e_oracle:.2e}, vs TrainStep {e_ts:.2e}')
    assert e_ts <= 1e-2, e_ts


@pytest.mark.parametrize('tag,skip,latent', [('base', True, None), ('film', False, 24), ('mag', False, None), ('magdb', True, None)])
def test_inference_unchanged(tag, skip, latent):
    """Eval mode and train mode under no_grad run the inference path: no graph, the same launches, and the values of the graph."""
    R, model, sd, c, audio, gt = _setup(tag, skip, latent)
    audio = audio.cuda()
    outs, counts = {}, {}
    for name in ('eval', 'no_grad', 'eval', 'no_grad'):        # the first round builds the packed weights
        _launches()
        if name == 'eval':
            o = model.eval()(audio, consistency=True)
            enc = model.encode(audio)
            dec = model.decode(enc[0], enc[1] if skip else None, transcribe=True)
        else:
            with torch.no_grad():
                o = model.train()(audio, consistency=True)
                enc = model.encode(audio)
                dec = model.decode(enc[0], enc[1] if skip else None, transcribe=True)
        counts[name] = _launches()
        flat = [t for t in o[:5]] + [enc[0]] + list(enc[1]) + [dec]
        assert all(t.grad_fn is None for t in flat), name
        outs[name] = flat
    assert counts['eval'] == counts['no_grad'], counts
    o = model.train()(audio, consistency=True)
    enc = model.encode(audio)
    dec = model.decode(enc[0], enc[1] if skip else None, transcribe=True)
    graph = [t for t in o[:5]] + [enc[0]] + list(enc[1]) + [dec]
    assert all(t.grad_fn is not None for t in graph)
    for a, b, g in zip(outs['eval'], outs['no_grad'], graph):
        assert torch.equal(a, b) and torch.equal(a, g.detach())


def test_frozen_encoder():
    """A frozen encoder gets no gradient, passes the consistency pass's data gradients through (the decoder's gradients are
    those of the unfrozen model, bit for bit) and skips its weight-gradient launches."""
    grads, launches = [], []
    for frozen in (False, True):
        R, model, sd, c, audio, gt = _setup('base', True)
        if frozen:
            model.encoder.requires_grad_(False)
        out = _reference_step(model, 'base', audio.cuda(), gt.cuda())
        _launches()
        out['total'].backward()
        launches.append(_launches())
        grads.append(_grads(model))
        if frozen:
            assert all(p.grad is None for p in model.encoder.parameters())
    dec = [k for k in grads[0] if k.startswith('decoder.')]
    assert dec and all(torch.equal(grads[0][k], grads[1][k]) for k in dec)
    assert torch.equal(grads[0]['skip_weights'], grads[1]['skip_weights'])
    print('backward launches unfrozen / frozen encoder', launches)
    assert launches[1] < launches[0], launches


@pytest.mark.parametrize('tag,latent', [('base', None), ('film', 24)])
def test_decode_input_gradients(tag, latent):
    """decode(latents, embeddings, transcribe) with skip connections: gradients to the latents, the embeddings and the parameters
    against the oracle's autograd."""
    R, model, sd, c, audio, gt = _setup(tag, True, latent)
    with torch.no_grad():
        lat0, emb0, _ = model.eval().encode(audio.cuda())
    g = torch.Generator().manual_seed(7)
    for transcribe in (False, True):
        lat = lat0.detach().cpu().requires_grad_(True)
        emb = [e.detach().cpu().requires_grad_(True) for e in emb0]
        lat_d = lat.detach().cuda().requires_grad_(True)
        emb_d = [e.detach().cuda().requires_grad_(True) for e in emb]
        model.train().zero_grad()
        y = model.decode(lat_d, emb_d, transcribe=transcribe)
        w = torch.randn(y.shape, generator=g)
        (y * w.cuda()).sum().backward()
        sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        (R.decode_variant_ref(tag, lat, sdg, c.n_bins, transcribe, emb) * w).sum().backward()
        got = dict(latents=lat_d.grad.cpu(), **{f'emb{i}': e.grad.cpu() for i, e in enumerate(emb_d)})
        want = dict(latents=lat.grad, **{f'emb{i}': e.grad for i, e in enumerate(emb)})
        got.update({k: p.grad.cpu() for k, p in model.named_parameters() if k.startswith('decoder.') or k.startswith('film_layer.')})
        want.update({k: v.grad for k, v in sdg.items() if k in got})
        err = _global_err(got, want)
        inputs = _global_err({k: got[k] for k in got if not k.startswith(('decoder.', 'film_layer.'))},
                             {k: want[k] for k in got if not k.startswith(('decoder.', 'film_layer.'))})
        print(f'{tag} transcribe={transcribe}: decode gradient rel-L2 {err:.2e}, latents + embeddings alone {inputs:.2e}')
        assert err <= 3e-2 and inputs <= 3e-2, (err, inputs)


def _close(got, want, tol=1e-5):
    got = got.detach().cpu()
    assert got.shape == want.shape
    assert float((got - want).abs().max()) <= tol * float(want.abs().max()), float((got - want).abs().max())


@pytest.mark.parametrize('tag', ['base', 'film', 'mag', 'magdb'])
def test_to_activations_gradient(tag):
    R, model, _, _, _, _ = _setup(tag, False, 24 if tag == 'film' else None)
    g = torch.Generator().manual_seed(11)
    C = 2 if tag in ('base', 'film') else 1
    x = torch.randn((2, C, 37, 64), generator=g)
    if tag == 'magdb':
        x = torch.sigmoid(x)
    w = torch.randn((2, 37, 64), generator=g)
    xr = x.clone().requires_grad_(True)
    (R.activations_variant_ref(tag, xr) * w).sum().backward()
    forms = [x.cuda()]
    if C == 2:
        forms.append(x.permute(0, 2, 3, 1).contiguous().cuda().permute(0, 3, 1, 2))      # a view of interleaved pairs, as forward returns
    for xd in forms:
        xd = xd.detach().requires_grad_(True)
        act = model.to_activations(xd)
        assert act.grad_fn is not None
        _close(act, R.activations_variant_ref(tag, x))
        (act * w.cuda()).sum().backward()
        _close(xd.grad, xr.grad)
    with torch.no_grad():
        assert model.to_activations(forms[0].detach().requires_grad_(True)).grad_fn is None


def _pair_forms(x):
    """(B, C, F, T) on the GPU as a contiguous tensor and as a permuted view of (B, F, T, C)."""
    return [x.cuda(), x.permute(0, 2, 3, 1).contiguous().cuda().permute(0, 3, 1, 2)]


def test_objective_gradients():
    from oracle import model_ref as R
    from timbre_trap_b200.framework import compute_consistency_loss, compute_reconstruction_loss, compute_transcription_loss
    g = torch.Generator().manual_seed(5)
    a, b, t = (torch.randn((3, 2, 41, 96), generator=g) for _ in range(3))
    ar, br, tr = (v.clone().requires_grad_(True) for v in (a, b, t))
    R.reconstruction_loss_ref(ar, br).backward()
    cs, ct = R.consistency_loss_ref(ar, br, tr)
    (cs * 0.7 + ct * 1.3).backward()
    for fa, fb, ft in [(x, y, z) for x in _pair_forms(a) for y in _pair_forms(b) for z in _pair_forms(t)]:
        va, vb, vt = (v.detach().requires_grad_(True) for v in (fa, fb, ft))
        compute_reconstruction_loss(va, vb).backward()
        cs, ct = compute_consistency_loss(va, vb, vt)
        (cs * 0.7 + ct * 1.3).backward()
        for got, want in ((va.grad, ar.grad), (vb.grad, br.grad), (vt.grad, tr.grad)):
            _close(got, want)
    # transcription: targets with exact ones (the positive class), partial values and zeros; an all-ones frame; a frame without ones
    est = torch.rand((2, 60, 80), generator=g)
    tgt = torch.zeros((2, 60, 80))
    tgt[:, 10] = 1.0
    tgt[:, 9] = tgt[:, 11] = 0.6
    tgt[0, 30:33, :40] = 1.0
    tgt[1, :, 5] = 1.0
    tgt[1, 10, 7] = 0.0
    for weighted in (False, True):
        er, tr_ = est.clone().requires_grad_(True), tgt.clone().requires_grad_(True)
        want = R.transcription_loss_ref(er, tr_, weighted)
        want.backward()
        ed, td = est.cuda().requires_grad_(True), tgt.cuda().requires_grad_(True)
        got = compute_transcription_loss(ed, td, weighted)
        np.testing.assert_allclose(float(got.detach()), float(want.detach()), rtol=1e-5)
        got.backward()
        _close(ed.grad, er.grad)
        _close(td.grad, tr_.grad)
        ed2 = est.cuda().requires_grad_(True)                   # the estimate alone
        compute_transcription_loss(ed2, tgt.cuda(), weighted).backward()
        assert torch.equal(ed2.grad, ed.grad)
    with torch.no_grad():
        assert compute_reconstruction_loss(a.cuda().requires_grad_(True), b.cuda()).grad_fn is None


@pytest.mark.parametrize('tag,skip,latent', [('base', True, None), ('film', True, 24)])
def test_autocast_has_no_effect(tag, skip, latent):
    """Under torch.autocast('cuda') (the reference's step, train.py:415) losses and gradients are bit-identical to those without."""
    results = []
    for amp in (False, True):
        R, model, sd, c, audio, gt = _setup(tag, skip, latent)              # a fresh model: its packed weights are built in the context
        with torch.autocast('cuda', enabled=amp):
            out = _reference_step(model, tag, audio.cuda(), gt.cuda())
            out['total'].backward()
        results.append(({k: v.detach() for k, v in out.items()}, _grads(model)))
    (l0, g0), (l1, g1) = results
    assert all(torch.equal(l0[k], l1[k]) for k in l0)
    assert set(g0) == set(g1) and all(torch.equal(g0[k], g1[k]) for k in g0)


def test_training_with_torch_optimizer_tracks_train_step():
    """Eight steps of the reference's loop (clip_grad_norm_(10) + torch.optim.AdamW) against eight TrainStep steps from the same
    weights: the same totals within 0.5 % per step, falling as in test_training_reduces_the_loss."""
    from timbre_trap_b200.framework.train import TrainStep
    R, model, sd, c, audio, gt = _setup('base')
    audio, gt = audio.cuda(), gt.cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=2e-3)
    api = []
    for _ in range(8):
        out = _reference_step(model, 'base', audio, gt)
        opt.zero_grad()
        out['total'].backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 10.0)
        opt.step()
        api.append(float(out['total'].detach()))
    R, model2, sd, c, _, _ = _setup('base')
    ts = TrainStep(model2, lr=2e-3)
    ref = [float(ts.step(audio, gt)['total']) for _ in range(8)]
    print('totals api', api, 'TrainStep', ref)
    np.testing.assert_allclose(api, ref, rtol=5e-3)
    assert api[-1] < 0.8 * api[0], api


def test_backward_pack_cache_bounded():
    """A torch optimizer updates the weights in place: the backward packs are replaced, not accumulated, and memory stays flat."""
    from timbre_trap_b200.framework import layer_grads as LG
    R, model, sd, c, audio, gt = _setup('film', True, 24)
    audio, gt = audio.cuda(), gt.cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    entries, mem = [], []
    params = list(model.parameters())
    for _ in range(5):
        out = _reference_step(model, 'film', audio, gt)
        opt.zero_grad()
        out['total'].backward()
        del out
        opt.step()
        torch.cuda.synchronize()
        entries.append(sum(len(LG._BW_PACKS.get(p, {})) for p in params))
        mem.append(torch.cuda.memory_allocated())
    print('backward packs per step', entries, 'allocated bytes', mem)
    assert entries[1:] == entries[:1] * 4, entries
    assert mem[4] <= mem[1], mem
