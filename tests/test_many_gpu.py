"""
TimbreTrap.transcribe_many / reconstruct_many / transcribe_and_reconstruct_many: clips of different lengths in one batched pass, each
result bit for bit what the one-clip call returns, with launches that follow the number of chunks and memory bounded by the group size.
"""
import numpy as np
import pytest
import torch

from tests.helpers import tonal_clip

pytestmark = pytest.mark.gpu

SMALL = dict(sample_rate=8000, n_octaves=6, bins_per_octave=12, secs_per_block=0.5)
BASE = dict(sample_rate=22050, n_octaves=9, bins_per_octave=60, secs_per_block=3)


def _build(cfg, latent, complexity, skip=False, seed=0, tag=None):
    from oracle import model_ref as R
    from timbre_trap_b200 import framework as FW
    cls = dict(film=FW.TimbreTrapFiLM, mag=FW.TimbreTrapMag, magdb=FW.TimbreTrapMagDB).get(tag, FW.TimbreTrap)
    model = cls(cfg['sample_rate'], cfg['n_octaves'], cfg['bins_per_octave'], cfg['secs_per_block'], latent_size=latent,
                model_complexity=complexity, skip_connections=skip)
    sd = R.init_state_dict(model.sliCQ.n_bins, latent, complexity, seed=seed, **({} if tag is None else dict(variant=tag)))
    if skip:
        sd['skip_weights'] = torch.tensor([0.9, 1.1, 0.8, 1.2, 0.7])
    model.load_state_dict(sd)
    return model.cuda().eval()


def _clips(model, lengths, seed):
    """Clips of the given lengths in a seeded shuffled order; one of shape (1, N) and one in float64 (converted as transcribe does)."""
    rng = np.random.default_rng(seed)
    lengths = [lengths[i] for i in rng.permutation(len(lengths))]
    sr = model.sliCQ.sample_rate
    clips = [(tonal_clip(n, sr, seed=seed + i)[0, 0] * float(rng.uniform(0.2, 1.0))).cuda() for i, n in enumerate(lengths)]
    clips[0] = clips[0].view(1, -1)
    clips[-1] = clips[-1].double()
    return clips


def _check_all(model, clips):
    one = [c.view(1, 1, -1) for c in clips]
    acts = model.transcribe_many(clips)
    wavs = model.reconstruct_many(clips)
    acts2, wavs2 = model.transcribe_and_reconstruct_many(clips)
    assert len(acts) == len(wavs) == len(acts2) == len(wavs2) == len(clips)
    for i, x in enumerate(one):
        a, w = model.transcribe(x)[0], model.reconstruct(x)[0]
        assert a.shape == acts[i].shape and w.shape == wavs[i].shape, (i, a.shape, acts[i].shape, w.shape, wavs[i].shape)
        assert torch.equal(acts[i], a), i
        assert torch.equal(wavs[i], w), i
        assert torch.equal(acts2[i], a), i
        assert torch.equal(wavs2[i], w), i
        pa, pw = model.transcribe_and_reconstruct(x)                  # the pair call against the two separate calls
        assert torch.equal(pa[0], a) and torch.equal(pw[0], w), i
    # one packed buffer per output kind
    assert len({a.untyped_storage().data_ptr() for a in acts2}) == 1
    assert len({w.untyped_storage().data_ptr() for w in wavs2}) == 1


@pytest.mark.parametrize('cfg,latent,complexity', [(SMALL, None, 1), (BASE, 128, 2)])
def test_many_equals_one_clip_calls(cfg, latent, complexity):
    model = _build(cfg, latent, complexity, seed=1)
    L = model.sliCQ.block_length
    # 1 sample, L - 1, L, L + 1, 2.6 L, and a clip of 7 chunks: longer than a chunk batch of 4, so batches cross clip boundaries and
    # the long clip spans several encoder / decoder launches; groups of at most 8 chunks split the list into several groups
    clips = _clips(model, [1, L - 1, L, L + 1, int(2.6 * L), 3 * L], seed=5)
    model.MAX_CHUNKS_PER_BATCH = 4
    model.MAX_CHUNKS_PER_GROUP = 8
    _check_all(model, clips)


@pytest.mark.parametrize('tag,skip,fuse', [('film', True, True), ('mag', False, True), ('magdb', True, True), (None, False, False)])
def test_many_variants_and_unfused(tag, skip, fuse):
    """FiLM with skips, Mag, MagDB with skips (their transcribe returns (2, F, T) per clip), and the un-fused convout + cross-fade."""
    model = _build(SMALL, 24, 2, skip=skip, seed=7, tag=tag)
    model.FUSE_CONVOUT_CROSSFADE = fuse
    L = model.sliCQ.block_length
    clips = _clips(model, [1, L + 1, int(2.6 * L), 3 * L], seed=9)
    model.MAX_CHUNKS_PER_BATCH = 4
    model.MAX_CHUNKS_PER_GROUP = 8
    _check_all(model, clips)
    if tag in ('mag', 'magdb'):
        assert model.transcribe_many(clips)[1].shape[0] == 2


def test_many_normalises_each_clip_by_its_own_peak():
    model = _build(SMALL, None, 1, seed=2)
    L = model.sliCQ.block_length
    loud = tonal_clip(2 * L + 5, SMALL['sample_rate'], seed=3)[0, 0].cuda()
    quiet = 1e-3 * tonal_clip(L - 7, SMALL['sample_rate'], seed=4)[0, 0].cuda()
    silent = torch.zeros(L + 3, device='cuda')
    wavs = model.reconstruct_many([quiet, silent, loud])
    for w, x in zip(wavs, (quiet, silent, loud)):
        assert abs(float(w.abs().max()) - 1.0) < 1e-6            # the model's biases make even silence decode to some sound
        assert torch.equal(w, model.reconstruct(x.view(1, 1, -1))[0])
    # reconstructions that ARE silent (convout zeroed) have peak 0: no divide, zeros back, no NaN
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    sd['decoder.convout.weight'].zero_()
    sd['decoder.convout.bias'].zero_()
    mute = _build(SMALL, None, 1, seed=2)
    mute.load_state_dict(sd)
    for w in mute.reconstruct_many([silent, loud]):
        assert not bool(torch.isnan(w).any()) and not bool(w.any())


def test_many_launches_follow_chunks_not_clips():
    """64 one-block clips (192 chunks) take no more library launches than one 95-block clip (191 chunks), plus a small constant."""
    from timbre_trap_b200 import _lib
    model = _build(SMALL, None, 1, seed=0)
    L = model.sliCQ.block_length
    g = torch.Generator(device='cuda').manual_seed(0)
    many = [torch.rand(L, device='cuda', generator=g) - 0.5 for _ in range(64)]
    one = [torch.rand(95 * L, device='cuda', generator=g) - 0.5]
    counts = []
    for clips in (many, one):
        model.transcribe_and_reconstruct_many(clips)          # warm-up: plans and packed weights
        torch.cuda.synchronize()
        _lib.lib().tt_launch_count(1)
        model.transcribe_and_reconstruct_many(clips)
        counts.append(int(_lib.lib().tt_launch_count(1)))
    assert counts[0] <= counts[1] + 4, counts


def test_many_peak_memory_is_bounded_by_the_group():
    """Doubling the number of equal clips raises peak allocation by the added outputs only (the stage buffers hold one group).  The
    1 MiB of slack is the caching allocator's: it hands out a cached block whole when less than 1 MiB of it would be left.  Without
    the grouping the 8 added clips would add 40 chunks of stage buffers, 11.8 MB."""
    model = _build(SMALL, None, 1, seed=0)
    L = model.sliCQ.block_length
    model.MAX_CHUNKS_PER_GROUP = 12                            # two 2-block clips (5 chunks each) per group
    g = torch.Generator(device='cuda').manual_seed(1)
    clips = [torch.rand(2 * L - 3, device='cuda', generator=g) - 0.5 for _ in range(16)]
    model.transcribe_and_reconstruct_many(clips[:2])          # warm-up
    peaks, out_bytes = [], []
    for k in (8, 16):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        acts, wavs = model.transcribe_and_reconstruct_many(clips[:k])
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
        out_bytes.append(sum(a.numel() for a in acts) * 4 + sum(w.numel() for w in wavs) * 4)
        del acts, wavs
    assert peaks[1] - peaks[0] <= out_bytes[1] - out_bytes[0] + 1024 * 1024, (peaks, out_bytes)


def test_many_validation():
    from timbre_trap_b200._lib import TimbreTrapB200Error
    model = _build(SMALL, None, 1, seed=0)
    L = model.sliCQ.block_length
    ok = torch.zeros(L, device='cuda')
    assert model.transcribe_many([]) == [] and model.reconstruct_many([]) == []
    assert model.transcribe_and_reconstruct_many([]) == ([], [])
    with pytest.raises(TimbreTrapB200Error):
        model.transcribe_many([ok, torch.zeros(L)])
    with pytest.raises(ValueError):
        model.transcribe_many([ok, torch.zeros(0, device='cuda')])
    with pytest.raises(ValueError):
        model.reconstruct_many([torch.zeros(2, L, device='cuda')])
    with pytest.raises(ValueError):
        model.transcribe_many([torch.zeros(1, 1, L, device='cuda')])
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            model.transcribe_many([ok, torch.zeros(L, device='cuda:1')])
