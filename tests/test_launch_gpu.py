"""
Every kernel runs with its tensors' device current: a model on cuda:1 computes the same values, bit for bit, whichever device is
current when it is called, and never launches with another device current; tensors on two devices are refused before any launch.
"""
import numpy as np
import pytest
import torch

from tests.helpers import tonal_clip

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two CUDA devices')]

SMALL = dict(sample_rate=8000, n_octaves=6, bins_per_octave=12, secs_per_block=0.5)
DEV = 'cuda:1'
# entry points that launch nothing; plans are also destroyed from _Plan.__del__, whenever an earlier test's model is collected
EXEMPT = ('tt_last_error', 'tt_version', 'tt_launch_count', 'tt_set_strip_rows', 'tt_cqt_plan_destroy')


class _CurrentDeviceCheck:
    """The loaded library, with a check before every call that cuda:1 is the current device; `calls` records what was forwarded."""

    def __init__(self, lib):
        self.lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if name in EXEMPT or name.endswith('_scratch_floats'):
            return fn

        def checked(*args):
            assert torch.cuda.current_device() == 1, f'{name} called with cuda:{torch.cuda.current_device()} current'
            self.calls.append(name)
            return fn(*args)
        return checked


@pytest.fixture
def checked_lib():
    from timbre_trap_b200 import _lib
    real = _lib.lib()
    _lib._lib = _CurrentDeviceCheck(real)
    try:
        yield _lib._lib
    finally:
        _lib._lib = real


def _model(tag, skip):
    from oracle import model_ref as R
    from timbre_trap_b200 import framework as FW
    cls = dict(base=FW.TimbreTrap, film=FW.TimbreTrapFiLM, mag=FW.TimbreTrapMag)[tag]
    model = cls(latent_size=24, model_complexity=1, skip_connections=skip, **SMALL)
    sd = R.init_state_dict(model.sliCQ.n_bins, 24, 1, seed=3, variant=tag)
    if skip:
        sd['skip_weights'] = torch.tensor([0.9, 1.1, 0.8, 1.2, 0.7])
    model.load_state_dict(sd)
    return model.to(DEV)


def _run():
    """The public calls on a SMALL model on cuda:1 -> {name: tensor or float}."""
    from timbre_trap_b200.framework import (TrainStep, compute_consistency_loss, compute_reconstruction_loss, compute_transcription_loss,
                                            frontend, postprocess as PP)
    out = {}
    model = _model('base', True)
    L, F, M = model.sliCQ.block_length, model.sliCQ.n_bins, model.sliCQ.max_window_length
    audio = tonal_clip(2 * L, SMALL['sample_rate'], seed=4, n_batch=3).to(DEV)
    gt = torch.zeros((2, F, 2 * M), device=DEV)
    gt[0, 10:13], gt[1, 20:23] = 1.0, 1.0

    model.eval()
    out['act'], out['wav'] = model.transcribe_and_reconstruct(audio)
    acts, wavs = model.transcribe_and_reconstruct_many([audio[0, 0], audio[1, 0, :L + 100], audio[2, 0, :300]])
    out.update({f'many_act{i}': a for i, a in enumerate(acts)}, **{f'many_wav{i}': w for i, w in enumerate(wavs)})
    tiled = model.forward_tiled(audio, consistency=True)
    out.update({f'tiled{i}': t for i, t in enumerate(tiled[:5])})

    for tag, skip in (('base', True), ('film', False)):
        ts = TrainStep(_model(tag, skip))
        res = ts.step(audio, gt)
        # the gradient norm is an atomic sum (its last bits vary between runs); the losses and gradients are fixed-order
        out.update({f'{tag}_step_{k}': v for k, v in res.items() if k != 'grad_norm'}, **{f'{tag}_step_grads': ts.flat_g})

    model = _model('mag', False).train()
    target = model.sliCQ.to_magnitude(model.sliCQ(audio)).unsqueeze(1)
    rec, _, trn, trn_rec, trn_scr, _ = model(audio, consistency=True)
    act = model.to_activations(trn)
    losses = [compute_reconstruction_loss(rec, target), compute_transcription_loss(act[:2], gt, True),
              *compute_consistency_loss(trn_rec[:2], trn_scr[:2], trn[:2])]
    sum(losses).backward()
    out.update({f'mag_loss{i}': v.detach() for i, v in enumerate(losses)})
    out.update({f'mag_grad_{k}': p.grad for k, p in model.named_parameters() if p.grad is not None})

    stereo = tonal_clip(3000, 16000, seed=5, n_batch=2)[:, 0].to(DEV)
    out['prepared'] = frontend.prepare_audio(stereo, 16000, SMALL['sample_rate'])
    out['pitches'] = frontend.multi_pitch_to_activations([np.array([220.0, 440.0]), np.array([]), np.array([330.0])],
                                                         model.sliCQ.get_midi_freqs(), device=DEV)
    out['sdr'] = frontend.signal_distortion_ratio(out['wav'], audio)
    a = out['act']
    out['peaks'] = PP.filter_non_peaks(a)
    out['threshold'] = PP.threshold(a, 0.3)
    est, ref = PP.activations_to_binary(a, 0.3, peaks_only=True), PP.activations_to_binary(a, 0.5)
    out['binary'] = est
    out['counts'] = PP.multipitch_counts(est, ref, 1)
    out.update({f'score_{k}': v for k, v in PP.multipitch_scores(est, ref, 1).items()})
    torch.cuda.synchronize(DEV)
    return out


def test_model_on_a_device_that_is_not_current(checked_lib):
    """cuda:0 current, everything on cuda:1: every launch runs with cuda:1 current and the results equal those of the same calls with
    cuda:1 current."""
    with torch.cuda.device(0):
        got = _run()
    n = len(checked_lib.calls)
    with torch.cuda.device(1):
        want = _run()
    assert n > 0 and checked_lib.calls[:n] == checked_lib.calls[n:2 * n], 'the two runs launched different kernels'
    assert got.keys() == want.keys()
    for k, w in want.items():
        if isinstance(w, torch.Tensor):
            assert got[k].device == torch.device(DEV), k
            torch.testing.assert_close(got[k], w, rtol=0, atol=0, equal_nan=True, msg=k)     # bit for bit
        else:
            assert got[k] == w, k


def test_tensors_on_two_devices_are_refused(checked_lib):
    from timbre_trap_b200.framework import ops
    x = torch.ones(64, dtype=torch.bfloat16, device='cuda:0')
    e = torch.ones(64, dtype=torch.bfloat16, device='cuda:1')
    with torch.cuda.device(1), pytest.raises(ValueError, match='one device'):
        ops.add_scaled(x, e, torch.ones((), device='cuda:0'))
    assert checked_lib.calls == []
