"""
framework.HostPipeline / TimbreTrap.transcribe_and_reconstruct(on_activations=...): host-to-host streaming must return exactly what
the one-shot device call returns - handing finished clips' activations over after every chunk batch and copying them out while the
next batch computes changes WHEN bytes move, not their values.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

SMALL = dict(sample_rate=8000, n_octaves=6, bins_per_octave=12, secs_per_block=0.5)


def _model(seed=5):
    from oracle import model_ref as R
    from timbre_trap_b200.framework import TimbreTrap
    model = TimbreTrap(SMALL['sample_rate'], SMALL['n_octaves'], SMALL['bins_per_octave'], SMALL['secs_per_block'], latent_size=None, model_complexity=1)
    model.load_state_dict(R.init_state_dict(model.sliCQ.n_bins, None, 1, seed=seed))
    return model.cuda().eval()


def _batches(model, n, clips, blocks=2):
    g = torch.Generator().manual_seed(11)
    L = model.sliCQ.block_length
    # different loudness per clip and per batch, so that a slice-local peak would show
    return [((torch.rand((clips, 1, blocks * L), generator=g) * 2 - 1) * torch.linspace(0.1, 1.0, clips).view(-1, 1, 1) * (0.5 + 0.5 * k / n)).pin_memory()
            for k in range(n)]


@pytest.mark.parametrize('max_chunks', [4, 5, 7, 256])
def test_early_activations_equal_whole(max_chunks):
    """The hook sees consecutive clip ranges covering the batch once, each holding the final activations at the time of the call
    (stream-ordered), whatever the chunk batch size (clips here have 5 chunks: batches end inside and between clips)."""
    model = _model()
    audio = _batches(model, 1, 7)[0].cuda()
    act, wav = model.transcribe_and_reconstruct(audio)
    model.MAX_CHUNKS_PER_BATCH = max_chunks
    seen = []
    act2, wav2 = model.transcribe_and_reconstruct(audio, on_activations=lambda lo, hi, a: seen.append((lo, hi, a.clone())))
    assert torch.equal(act2, act) and torch.equal(wav2, wav)
    assert seen[0][0] == 0 and seen[-1][1] == 7 and all(a[1] == b[0] for a, b in zip(seen, seen[1:]))
    assert (len(seen) > 1) == (max_chunks < 35)
    assert torch.equal(torch.cat([a for _, _, a in seen]), act)


def test_transcribe_and_reconstruct_does_not_wait_for_the_device():
    """No host synchronisation in the call, with or without the early hand-over: HostPipeline keeps two steps in flight only if
    submitting one does not wait for the other."""
    model = _model()
    audio = _batches(model, 1, 3)[0].cuda()
    model.MAX_CHUNKS_PER_BATCH = 4
    hook = lambda lo, hi, a: None
    model.transcribe_and_reconstruct(audio, on_activations=hook)       # warm-up: plans, packed weights, windows
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        model.transcribe_and_reconstruct(audio)
        model.transcribe_and_reconstruct(audio, on_activations=hook)
    finally:
        torch.cuda.set_sync_debug_mode('default')


@pytest.mark.parametrize('early,depth,max_chunks', [(False, 2, 256), (True, 3, 256), (True, 3, 7), (True, 2, 11)])
def test_pipeline_returns_the_device_results(early, depth, max_chunks):
    from timbre_trap_b200.framework import HostPipeline
    model = _model()
    batches = _batches(model, 5, 6)
    want = [tuple(t.cpu() for t in model.transcribe_and_reconstruct(b.cuda())) for b in batches]
    model.MAX_CHUNKS_PER_BATCH = max_chunks
    pipe = HostPipeline(model, depth=depth, early=early)
    in_flight, got = [], []
    for b in batches:
        in_flight.append(pipe.submit(b))
        if len(in_flight) > depth - 1:
            got.append(tuple(t.clone() for t in pipe.collect(in_flight.pop(0))))
    got += [tuple(t.clone() for t in pipe.collect(k)) for k in in_flight]
    assert len(got) == len(want)
    for (a, w), (a0, w0) in zip(got, want):
        assert torch.equal(a, a0) and torch.equal(w, w0)
    h2d, d2h = pipe.bytes_per_step(batches[0])
    assert h2d == batches[0].numel() * 4 and d2h == (want[0][0].numel() + want[0][1].numel()) * 4


def test_pipeline_overwritten_ticket_is_an_error():
    from timbre_trap_b200.framework import HostPipeline
    model = _model()
    b = _batches(model, 1, 2)[0]
    pipe = HostPipeline(model, depth=2)
    first = pipe.submit(b)
    pipe.submit(b)
    pipe.submit(b)                                   # reuses the first slot
    with pytest.raises(ValueError):
        pipe.collect(first)


def test_pipeline_changing_batch_shape():
    from timbre_trap_b200.framework import HostPipeline
    model = _model()
    model.MAX_CHUNKS_PER_BATCH = 6
    pipe = HostPipeline(model, depth=2)
    for clips in (4, 6, 4):
        b = _batches(model, 1, clips)[0]
        act, wav = pipe.collect(pipe.submit(b))
        a0, w0 = model.transcribe_and_reconstruct(b.cuda())
        assert torch.equal(act, a0.cpu()) and torch.equal(wav, w0.cpu())
