"""
Throughput of a corpus of clips of different lengths, three ways (base model: 9 oct x 60 bpo, 22.05 kHz, latent 128, complexity 2,
random init):

  (a) loop   one TimbreTrap.transcribe_and_reconstruct call per clip
  (b) many   TimbreTrap.transcribe_and_reconstruct_many over the whole corpus
  (c) padded clips sorted by length, batches of pad-to-longest (at most --padded-chunks chunks per batch)

    python scripts/time_many.py OUTDIR [--minutes 30] [--reps 3] [--seed 0]

Seeded corpus: log-normal lengths clipped to [1 s, 120 s] until the total reaches --minutes.  Each approach is warmed up once over
the whole corpus, then timed --reps times with CUDA events around the pass and a device synchronise; the median is reported as
audio-s/s, with the chunks each approach computed.  (a) and (b) are also compared bit for bit.  Writes OUTDIR/time_many.json with the
GPU's name, power limit and SM clocks read in the same run.
"""

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SR, N_OCT, BPO, SECS, LATENT, COMPLEXITY = 22050, 9, 60, 3, 128, 2


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        row = subprocess.run(['nvidia-smi', '-i', str(torch.cuda.current_device()), f'--query-gpu={q}', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(','), [v.strip() for v in row.split(',')]))
    except Exception as e:               # the measurement stands without it, but says so
        return dict(name=torch.cuda.get_device_name(), error=f'nvidia-smi: {e}')


def corpus(minutes, seed, device):
    rng = np.random.default_rng(seed)
    lengths = []
    while sum(lengths) < minutes * 60 * SR:
        secs = float(np.clip(rng.lognormal(np.log(20.0), 1.0), 1.0, 120.0))
        lengths.append(int(secs * SR))
    g = torch.Generator(device=device).manual_seed(seed)
    return [torch.rand(n, device=device, generator=g) * 2 - 1 for n in lengths]


def timed(fn, reps):
    fn()                                                    # warm-up over the whole corpus
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return sorted(ms)[len(ms) // 2], ms, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('outdir')
    ap.add_argument('--minutes', type=float, default=30.0)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--padded-chunks', type=int, default=768, help='most chunks per pad-to-longest batch (c)')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('time_many.py measures on the GPU; no CUDA device found')
    from timbre_trap_b200.framework import TimbreTrap
    device = torch.device('cuda')
    torch.manual_seed(args.seed)
    model = TimbreTrap(SR, N_OCT, BPO, SECS, latent_size=LATENT, model_complexity=COMPLEXITY).to(device).eval()
    L = model.sliCQ.block_length
    clips = corpus(args.minutes, args.seed, device)
    lengths = np.array([c.numel() for c in clips])
    blocks = -(-lengths // L)
    audio_s = float(lengths.sum()) / SR

    def loop():
        return [model.transcribe_and_reconstruct(c.view(1, 1, -1)) for c in clips]

    def many():
        return model.transcribe_and_reconstruct_many(clips)

    order = np.argsort(lengths, kind='stable')
    batches, cur = [], []
    for i in order:                                          # ascending: the last clip of a batch is its longest
        if cur and (len(cur) + 1) * (2 * blocks[i] + 1) > args.padded_chunks:
            batches.append(cur)
            cur = []
        cur.append(int(i))
    batches.append(cur)
    padded_batches = []
    for b in batches:
        n = int(lengths[b[-1]])
        x = torch.zeros((len(b), 1, n), device=device)
        for j, i in enumerate(b):
            x[j, 0, :lengths[i]] = clips[i]
        padded_batches.append(x)

    def padded():
        return [model.transcribe_and_reconstruct(x) for x in padded_batches]

    chunks = dict(loop=int((2 * blocks + 1).sum()), many=int((2 * blocks + 1).sum()),
                  padded=int(sum(len(b) * (2 * blocks[b[-1]] + 1) for b in batches)))
    info = gpu_info()
    results = {}
    outs = {}
    for name, fn in (('loop', loop), ('many', many), ('padded', padded)):
        med, ms, out = timed(fn, args.reps)
        results[name] = dict(median_ms=med, ms=ms, audio_s_per_s=audio_s / (med / 1e3), chunks=chunks[name],
                             launches_per_pass=None)
        if name != 'padded':
            outs[name] = out
        print(f'{name:7s} {med:10.1f} ms  {audio_s / (med / 1e3):9.0f} audio-s/s  {chunks[name]} chunks', flush=True)
        del out
    from timbre_trap_b200 import _lib
    for name, fn in (('loop', loop), ('many', many), ('padded', padded)):
        _lib.lib().tt_launch_count(1)
        fn()
        results[name]['launches_per_pass'] = int(_lib.lib().tt_launch_count(1))
    acts_b, wavs_b = outs['many']
    identical = all(torch.equal(a[0][0], acts_b[i]) and torch.equal(a[1][0], wavs_b[i]) for i, a in enumerate(outs['loop']))
    res = dict(gpu=info, model=dict(sample_rate=SR, n_octaves=N_OCT, bins_per_octave=BPO, secs_per_block=SECS, latent_size=LATENT,
                                   model_complexity=COMPLEXITY),
               corpus=dict(seed=args.seed, clips=len(clips), audio_s=audio_s, min_s=float(lengths.min()) / SR,
                           max_s=float(lengths.max()) / SR, median_s=float(np.median(lengths)) / SR, blocks=int(blocks.sum())),
               padded_batches=len(batches), reps=args.reps, results=results, many_equals_loop_bit_for_bit=bool(identical),
               max_chunks_per_batch=model.MAX_CHUNKS_PER_BATCH, max_chunks_per_group=model.MAX_CHUNKS_PER_GROUP)
    os.makedirs(args.outdir, exist_ok=True)
    with open(os.path.join(args.outdir, 'time_many.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
