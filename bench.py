"""
Benchmark of the Timbre-Trap hot path on B200 (contract: see the round prompt / DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--blocks 256] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[2], the configuration the audio-s/s metric is quoted on): transcribe + reconstruct of a
batch of 256 synthetic 3 s blocks (768 audio-seconds) per GPU with the base model (9 oct x 60 bpo, 22.05 kHz, latent
128, complexity 2, random init, bf16 convs / fp32 CQT).  One step = TimbreTrap.transcribe_and_reconstruct on the
whole batch: chunking (50 % overlap -> 3 chunks per block), CQT analysis, encoder (once), decoder (twice), Hann
cross-fade, tanh|.| activations, CQT synthesis + peak normalise.  Multi-GPU: blocks are sharded across ranks (weak
scaling, no data-path collective; one scalar MAX all-reduce for the reference's global peak normalise).

Printed by rank 0: ONE JSON line (metric/value/e2e/roofline/cpu_baseline/clocks/...).  `--impl reference` times the CPU
restatement of the reference path (oracle/, the reference itself is pure Python + a missing third-party CQT and does not
exist on the GPU box) on the host cores, on a bounded sample of the same workload.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

SR, N_OCT, BPO, SECS, LATENT, COMPLEXITY = 22050, 9, 60, 3, 128, 2
L, F, M = 66150, 540, 1024
METRIC = 'audio-sec/sec transcribe+reconstruct'
UNIT = 'audio-s/s'


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p['hbm_gbs'], bf16_burst=p['bf16_tflops'], bf16_sustained=p['bf16_tflops_sustained'], source='measured')
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source='fallback')


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=int(self.rows[0][1]) if self.rows else None,
                    samples=len(sm), reasons=sorted(reasons))


def synthetic_audio(n_blocks, seed, device='cpu', pin=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((n_blocks, 1, L), generator=g) * 2 - 1
    if pin:
        x = x.pin_memory()
    return x.to(device) if device != 'cpu' else x


class TorchReference:
    """
    The reference's own code path restated with library calls only, on any torch device: the oracle's functional model
    (oracle/model_ref.py: F.conv2d / F.conv_transpose2d / F.elu) with the NSGT as torch.fft calls on the oracle's tables (what
    cqt_pytorch does), run as the reference runs it - model.transcribe(audio) then model.reconstruct(audio), each a sequential loop
    over the chunk positions with the whole batch per iteration (modules.py:247-263).
      device cpu  (fp32, all host threads): the CPU arm - `--impl reference` and `cpu_baseline`
      device cuda (bf16 autocast: cuFFT + cuDNN + ATen): `gpu_eager_baseline`, a DIAGNOSTIC ANCHOR (SURVEY.md section 2.1)
    Never on the product path; bench.py only.
    """

    def __init__(self, device):
        from oracle import model_ref as R
        self.R = R
        self.device = torch.device(device)
        cq = R.CQTRef(N_OCT, BPO, SR, SECS)
        t = cq.nsgt.tables
        self.block_length, self.max_window_length, self.n_bins = cq.block_length, cq.max_window_length, cq.n_bins
        self.idx = torch.from_numpy(t.idx).to(device)
        self.win = torch.from_numpy(t.win).float().to(device)
        self.win_inv = torch.from_numpy(t.win_inv).float().to(device)
        self.sd = {k: v.to(device) for k, v in R.init_state_dict(F, LATENT, COMPLEXITY, seed=0).items()}
        self.to_magnitude = R.CQTRef.to_magnitude

    def pad_to_block_length(self, audio):
        return torch.nn.functional.pad(audio, (0, -audio.size(-1) % self.block_length))

    def get_expected_frames(self, n):
        import math
        return math.ceil((n / self.block_length) * self.max_window_length)

    def __call__(self, audio):                   # CQT.forward: (B, 1, n L) -> (B, 2, F, n M)
        B, _, N = audio.shape
        n = N // self.block_length
        spec = torch.fft.fft(audio.float().reshape(B, n, self.block_length))
        c = torch.fft.ifft(spec[..., self.idx] * self.win)                     # (B, n, F, M)
        c = c.permute(0, 2, 1, 3).reshape(B, self.n_bins, n * self.max_window_length)
        return torch.view_as_real(c).permute(0, 3, 1, 2)

    def decode(self, coeffs):                    # CQT.decode incl. the global peak normalise and its host sync
        B, _, Fq, T = coeffs.shape
        n = T // self.max_window_length
        c = torch.view_as_complex(coeffs.float().permute(0, 2, 3, 1).contiguous()).reshape(B, Fq, n, self.max_window_length).permute(0, 2, 1, 3)
        taps = torch.fft.fft(c) * self.win_inv
        Y = torch.zeros((B, n, self.block_length), dtype=taps.dtype, device=taps.device)
        Y.scatter_add_(-1, self.idx.reshape(1, 1, -1).expand(B, n, -1), taps.reshape(B, n, -1))
        audio = torch.fft.ifft(Y).real.reshape(B, 1, n * self.block_length)
        peak = audio.abs().max()
        if peak:
            audio = audio / peak
        return audio

    def step(self, audio):
        """chunked_inference (modules.py:204-269) twice, exactly the oracle's loop but with device-side buffers."""
        R, hop, Mw = self.R, self.block_length // 2, self.max_window_length
        window = R.hann_sym(Mw).to(self.device)
        outs = []
        with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16, enabled=self.device.type == 'cuda'):
            for transcribe in (True, False):
                x = torch.nn.functional.pad(self.pad_to_block_length(audio), [hop, hop])
                n_chunks = (x.size(-1) - hop) // hop
                out = torch.zeros((audio.size(0), 2, self.n_bins, self.get_expected_frames(x.size(-1))), device=self.device)
                for i in range(n_chunks):
                    piece = x[..., i * hop: i * hop + self.block_length]
                    out[..., i * Mw // 2: i * Mw // 2 + Mw] += window * R.inference_ref(piece, self.sd, self, transcribe).float()
                out = out[..., Mw // 2: -Mw // 2]
                outs.append(torch.tanh(self.to_magnitude(out)) if transcribe else self.decode(out))
        return outs


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path (model.transcribe(audio); model.reconstruct(audio), modules.py:292-336)
# ---------------------------------------------------------------------------------------------------------------
def cpu_reference_step(state, n_blocks):
    audio = synthetic_audio(n_blocks, seed=0)
    t0 = time.perf_counter()
    state.step(audio)
    return time.perf_counter() - t0


def cpu_state():
    torch.set_num_threads(os.cpu_count() or 1)
    return TorchReference('cpu')


WORKLOAD = ('BASELINE.json configs[2]: transcribe+reconstruct, 256 x 3 s blocks per GPU, base model '
            '(9 oct x 60 bpo, 22.05 kHz, latent 128, complexity 2), random init')


CPU_BLOCKS = 8        # blocks per CPU step: the reference's chunk loop runs the whole batch through each chunk position


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2] if len(xs) % 2 else 0.5 * (xs[len(xs) // 2 - 1] + xs[len(xs) // 2])


def run_reference(args, rank):
    if rank != 0:
        return
    state = cpu_state()
    n_blocks = CPU_BLOCKS                     # bounded sample of the 256-block batch: 8 blocks per step, all host threads
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_reference_step(state, n_blocks)
    times = [cpu_reference_step(state, n_blocks) for _ in range(args.steps)]
    per_step = median(times)                  # BASELINE.md section 4: median of >= 5 runs after one warm-up
    value = n_blocks * SECS / per_step
    cores = torch.get_num_threads()
    line = dict(metric=METRIC, value=value, unit=UNIT, impl='reference', n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=per_step * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
                config=dict(workload=WORKLOAD, sample=f'bounded sample of that workload: a batch of {n_blocks} x 3 s blocks per step on the host '
                                                      'CPU (the reference\'s sequential chunk loop over the batch), median step time'),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind='port',
                                  sample=f'{args.steps} steps x {n_blocks} block(s) of 3 s; oracle/model_ref.py convs + a torch.fft NSGT on the oracle tables (the '
                                         'reference is pure Python with an un-vendored CQT dependency; /root/reference is absent on the GPU box)'),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    emit(line)


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def time_kernel(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters          # ms


def synthetic_targets(n_items, n_frames, seed):
    """Multi-pitch targets in the manner of PitchDataset.multi_pitch_to_activations (datasets/PitchDataset.py:233-307): exact 1.0
    at a few bins per frame held for >= 50 frames, Gaussian-blurred neighbours (sigma = 1 bin), clipped to [0, 1]."""
    import numpy as np
    rng = np.random.default_rng(seed)
    gt = np.zeros((n_items, F, n_frames), dtype=np.float32)
    blur = np.exp(-0.5 * np.arange(-3, 4) ** 2)
    for b in range(n_items):
        t = 0
        while t < n_frames:
            hold = int(rng.integers(50, 400))
            for k in rng.integers(30, F - 30, size=int(rng.integers(1, 7))):
                for o, g in zip(range(-3, 4), blur):
                    gt[b, k + o, t:t + hold] = np.maximum(gt[b, k + o, t:t + hold], g)
            t += hold
    return torch.from_numpy(gt)


DUMP_ELEMENTS = 12 << 20      # float32 values --dump-outputs writes in all (48 MiB), shared equally by the outputs


def dump_outputs(out_dir, outputs):
    """Writes each tensor of `outputs` (name -> tensor) as out_dir/<name>.npy in float32.  One that fits its share of DUMP_ELEMENTS is
    written whole, in its own shape; a larger one as a 1-D array of its elements at sorted flat indices drawn without replacement by a
    generator of fixed seed from its element count alone, so two runs with the same arguments write the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_ELEMENTS // len(outputs)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > share:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), share, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f'{name}.npy'), t.float().cpu().numpy())


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from timbre_trap_b200 import _lib
    from timbre_trap_b200.framework import HostPipeline, TimbreTrap, TrainStep

    device = torch.device('cuda', local_rank)
    torch.cuda.set_device(device)
    group = None
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
        group = dist.group.WORLD

    torch.manual_seed(0)
    model = TimbreTrap(SR, N_OCT, BPO, SECS, latent_size=LATENT, model_complexity=COMPLEXITY).to(device).eval()
    n_blocks = args.blocks
    host_audio = synthetic_audio(n_blocks, seed=1000 + rank, pin=True)
    dev_audio = host_audio.to(device)
    pk = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        return model.transcribe_and_reconstruct(dev_audio, group=group)

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- device-resident arm ----
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.lib().tt_launch_count(1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps - 1):
        step_resident()
    last = step_resident()                      # held past the loop only: the earlier steps' outputs are freed as before
    b.record()
    barrier()
    launches = int(_lib.lib().tt_launch_count(1))
    ms_total = max_over_ranks(a.elapsed_time(b))
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(activations=last[0], audio=last[1]))
    del last
    ms_step = ms_total / args.steps
    value = world * n_blocks * SECS / (ms_step * 1e-3)
    # whole-step arithmetic against the SUSTAINED bf16 peak: 3 chunks per block, encoder once + decoder twice per chunk
    step_flops = 3 * n_blocks * 28.12e9
    step_tensor_frac = step_flops / (ms_step * 1e-3) / 1e12 / pk['bf16_sustained']

    # ---- end-to-end arm: pinned host audio in, pinned host results out, EVERY step, through framework.HostPipeline (copy-in /
    # compute / copy-out streams, double-buffered pinned outputs: the read-back of step k overlaps the compute of step k+1) ----
    pipe = HostPipeline(model, device, depth=3, group=group, early=not args.no_early)
    near = pipe.pinned_empty(host_audio.shape)          # the caller's batches, pinned on the GPU's own NUMA node like the outputs
    near.copy_(host_audio)
    host_audio = near
    for _ in range(max(len(pipe.slots), args.warmup // 2)):     # every buffer set once: pinned allocations are not part of a step
        pipe.collect(pipe.submit(host_audio))
    barrier()
    t0 = time.perf_counter()
    in_flight = []
    for _ in range(args.steps):
        in_flight.append(pipe.submit(host_audio))
        if len(in_flight) > 2:                                  # two steps stay enqueued: the host never waits on a read-back to launch
            pipe.collect(in_flight.pop(0))
    for k in in_flight:
        pipe.collect(k)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    barrier()
    h2d, d2h = pipe.bytes_per_step(host_audio)
    e2e = dict(value=world * n_blocks * SECS / (e2e_ms * 1e-3), unit=UNIT, ms_per_step=e2e_ms, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
               how='framework.HostPipeline: H2D of the step\'s audio, transcribe_and_reconstruct, D2H of activations + audio into pinned '
                   'buffers on copy streams, three buffer sets / two steps in flight, finished clips\' activations leave after every chunk batch while '
                   'the next one computes; wall clock from the first submit to the last result on the host')
    del pipe
    torch.cuda.empty_cache()

    # ---- BASELINE.json configs[3]: the loss step, batch 8 x 9 s per GPU, data-parallel (one flat-bucket NCCL all-reduce) ----
    train = None
    if not args.no_train:
        tb = 8
        g = torch.Generator().manual_seed(200 + rank)
        t_audio = (torch.rand((tb, 1, 3 * L), generator=g) * 2 - 1).to(device)
        t_gt = synthetic_targets(tb, 3 * M, seed=300 + rank).to(device)
        tmodel = TimbreTrap(SR, N_OCT, BPO, SECS, latent_size=LATENT, model_complexity=COMPLEXITY).to(device)
        ts = TrainStep(tmodel, group=group)
        for _ in range(3):
            res = ts.step(t_audio, t_gt)
        barrier()
        a.record()
        n_train = 5
        for _ in range(n_train):
            res = ts.step(t_audio, t_gt)
        b.record()
        barrier()
        t_ms = max_over_ranks(a.elapsed_time(b)) / n_train
        ar_us = None
        if world > 1:
            flat = torch.zeros(614490, device=device)
            ar_us = 1e3 * max_over_ranks(time_kernel(lambda: dist.all_reduce(flat, group=group), iters=20))
        train = dict(workload='BASELINE.json configs[3]: loss step (reconstruction + transcription + consistency), base model, batch 8 x 9 s per GPU',
                     ms_per_step=t_ms, audio_s_per_s=world * tb * 9 / (t_ms * 1e-3), tflops=4.05 / (t_ms * 1e-3),
                     frac_of_sustained_bf16=4.05 / (t_ms * 1e-3) / pk['bf16_sustained'], allreduce_us=ar_us, allreduce_bytes=614490 * 4,
                     total_loss=float(res['total']), grad_norm=float(res['grad_norm']))
        del ts, tmodel, t_audio, t_gt, res
        torch.cuda.empty_cache()

    # ---- BASELINE.json configs[4]: ONE 1-hour clip (1200 blocks -> 2401 overlapped chunks) sharded by blocks over the ranks ----
    hour = None
    if not args.no_hour:
        gh = torch.Generator().manual_seed(77)
        clip = ((torch.rand((1, 1, 1200 * L), generator=gh) * 2 - 1) * 0.5).to(device)      # every rank holds the clip
        for _ in range(1):
            model.transcribe_sharded(clip, group=group)
            model.transcribe_and_reconstruct_sharded(clip, group=group)
        barrier()
        n_hour = 2
        a.record()
        for _ in range(n_hour):
            h_act = model.transcribe_sharded(clip, group=group)
        b.record()
        barrier()
        h_ms_t = max_over_ranks(a.elapsed_time(b)) / n_hour
        a.record()
        for _ in range(n_hour):
            h_act, h_wav = model.transcribe_and_reconstruct_sharded(clip, group=group)
        b.record()
        barrier()
        h_ms = max_over_ranks(a.elapsed_time(b)) / n_hour
        hour = dict(workload='BASELINE.json configs[4]: one 3600 s clip (1200 blocks -> 2401 overlapped chunks) sharded by contiguous block ranges '
                             'over the ranks with half-block halos, all_gather of the frames (and one scalar MAX all-reduce for the audio)',
                    transcribe_ms=h_ms_t, transcribe_audio_s_per_s=3600.0 / (h_ms_t * 1e-3),
                    transcribe_and_reconstruct_ms=h_ms, transcribe_and_reconstruct_audio_s_per_s=3600.0 / (h_ms * 1e-3),
                    activations=list(h_act.shape), audio_out=list(h_wav.shape))
        del clip, h_act, h_wav
        torch.cuda.empty_cache()

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel family: the fused residual-block kernel (res_rs_kernel, ~60 % of the step).  Every
        # instance is HBM-bound un-fused (arithmetic intensity 17..136 FLOP/B against a ridge of ~210).  `roofline` reports the
        # first-stage instance (C = 4, packed layout, the largest tensors) against the measured copy bandwidth, `family_frac` all
        # twelve (stage, dilation) instances of the model timed alone back to back, and `roofline_tensor` the C = 32 instance
        # against the measured bf16 burst peak (the north star's tensor-pipe view).
        n_chunks = min(3 * n_blocks, model.MAX_CHUNKS_PER_BATCH)
        fam_bytes = fam_ms = 0.0
        per_instance = {}
        shapes = {4: (n_chunks, F, M, 4), 8: (n_chunks, 1, 269, M, 8), 16: (n_chunks, 2, 133, M, 8), 32: (n_chunks, 4, 65, M, 8)}
        for blk_e, c in ((model.encoder.block1, 4), (model.encoder.block2, 8), (model.encoder.block3, 16), (model.encoder.block4, 32)):
            x = torch.randn(shapes[c], device=device).to(torch.bfloat16)
            y = torch.empty_like(x)
            for rb in (blk_e.block1, blk_e.block2, blk_e.block3):
                ms = time_kernel(lambda: rb.forward_c8(x, out=y), iters=10)
                h = x.shape[1] if c == 4 else x.shape[2]
                nbytes = 2.0 * n_chunks * c * h * M * 2                    # read x + write y, un-padded channels, bf16
                per_instance[(c, rb.dilation)] = (ms, nbytes)
                fam_bytes += nbytes
                fam_ms += ms
            del x, y
        ms_4, bytes_4 = per_instance[(4, 1)]
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'r02_res_rs_c4_traffic.json')
        if os.path.exists(tpath):
            t = json.load(open(tpath))
            traffic = t['dram_bytes_per_launch'] * (n_chunks / t['chunks'])
        roofline = dict(kernel='res_rs_kernel<2,16,1,4> (fused ResidualConv2dBlock, C=4 packed layout folded to 4 frames per GEMM row, dilation 1, H=540)', bound='hbm',
                        achieved=bytes_4 / (ms_4 * 1e-3) / 1e9, peak=pk['hbm'], unit='GB/s', frac=bytes_4 / (ms_4 * 1e-3) / 1e9 / pk['hbm'],
                        traffic=traffic, peak_source=f"{pk['source']} HBM copy bandwidth", us_per_launch=ms_4 * 1e3,
                        bytes_per_launch=bytes_4, chunks_per_launch=n_chunks,
                        family_frac=fam_bytes / (fam_ms * 1e-3) / 1e9 / pk['hbm'],
                        family=f'all 12 (stage, dilation) instances of res_rs_kernel in the model, {fam_bytes / 1e9:.1f} GB in {fam_ms:.2f} ms',
                        step_tensor_frac=step_tensor_frac,
                        step_tensor=f'whole step: {step_flops / 1e12:.1f} TFLOP (3 chunks per block x 28.12 GFLOP) in {ms_step:.1f} ms against the '
                                    f"{pk['source']} SUSTAINED bf16 peak {pk['bf16_sustained']} TFLOP/s")
        ms_k, _ = per_instance[(32, 2)]
        flops = 2.0 * (9 * 32 * 32 + 32 * 32) * 65 * M * n_chunks
        achieved = flops / (ms_k * 1e-3) / 1e12
        roofline_tensor = dict(kernel='res_rs_kernel<4,32,2,0> (fused ResidualConv2dBlock, C=32, dilation 2, H=65)', bound='tensor',
                               achieved=achieved, peak=pk['bf16_burst'], unit='TFLOP/s', frac=achieved / pk['bf16_burst'],
                               peak_source=f"{pk['source']} bf16 burst (kernel timed alone)", us_per_launch=ms_k * 1e3,
                               flops_per_launch=flops, hbm_gbs=per_instance[(32, 2)][1] / (ms_k * 1e-3) / 1e9)
        # ---- CQT forward / inverse against the HBM roofline (BASELINE.json configs[1]: 1024 blocks) ----
        cq = {}
        nb = 1024
        big = synthetic_audio(nb, seed=7, device=device)
        coeffs = model.sliCQ.encode_interleaved(big)
        bytes_dir = nb * (4 * L + 8 * F * M)
        for name, fn in (('forward', lambda: model.sliCQ.encode_interleaved(big)),
                         ('inverse', lambda: model.sliCQ.decode_raw(coeffs.permute(0, 3, 1, 2), normalise=True))):
            ms = time_kernel(fn, iters=5)
            cq[name] = dict(ms=ms, achieved=bytes_dir / (ms * 1e-3) / 1e9, peak=pk['hbm'], unit='GB/s',
                            frac=bytes_dir / (ms * 1e-3) / 1e9 / pk['hbm'], bytes=bytes_dir)
        cq['round_trip_audio_s_per_s'] = nb * SECS / ((cq['forward']['ms'] + cq['inverse']['ms']) * 1e-3)
        cq['workload'] = 'BASELINE.json configs[1]: 1024 x 3 s blocks, 540 bins, fp32; whole path (all kernels of the direction)'
        del big, coeffs
        torch.cuda.empty_cache()

        # ---- diagnostic anchor: the reference's own code path given a GPU (cuFFT + cuDNN + ATen, bf16 autocast), same batch ----
        eager = None
        if world == 1 and not args.no_eager:
            try:
                ref = TorchReference(device)
                ref.step(dev_audio[:8])
                torch.cuda.synchronize()
                ms_e = time_kernel(lambda: ref.step(dev_audio), iters=2, warm=1)
                eager = dict(value=n_blocks * SECS / (ms_e * 1e-3), unit=UNIT, ms_per_step=ms_e,
                             what='oracle/model_ref.py on CUDA under bf16 autocast (cuDNN convs, ATen element-wise) + torch.fft NSGT (cuFFT), '
                                  'model.transcribe then model.reconstruct as sequential chunk loops over the same 256-block batch; '
                                  'diagnostic anchor, not the reference arm')
                del ref
            except Exception as exc:                      # an anchor must not take the bench down (e.g. out of memory)
                eager = dict(unavailable=f'{type(exc).__name__}: {exc}'[:200])
            torch.cuda.empty_cache()

        cpu = None
        if world == 1 and not args.no_cpu:
            state = cpu_state()
            cpu_reference_step(state, CPU_BLOCKS)
            times = []
            t_start = time.perf_counter()
            while len(times) < 3 or (time.perf_counter() - t_start < 15 and len(times) < 7):
                times.append(cpu_reference_step(state, CPU_BLOCKS))
            v = CPU_BLOCKS * SECS / median(times)
            cpu = dict(value=v, unit=UNIT, cores=torch.get_num_threads(), kind='port',
                       sample=f'median of {len(times)} x (transcribe + reconstruct of a batch of {CPU_BLOCKS} x 3 s blocks, sequential 3-chunk '
                              'loops over the batch): oracle/model_ref.py convs + a torch.fft NSGT on the oracle tables, fp32, all host threads')

        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=ms_step,
                    higher_is_better=True, scaling='weak', vs_baseline=None, dtype='bf16 convs (fp32 accumulate), fp32 CQT',
                    data='synthetic', impl='ours',
                    config=dict(workload=WORKLOAD,
                                blocks_per_gpu=n_blocks, chunks_per_gpu=3 * n_blocks, parallelism=f'dp{world} (block sharding)',
                                l2='working set per step ~40 GB >> 126 MB L2; no explicit flush'),
                    e2e=e2e, gpu_launches=launches, roofline=roofline, roofline_tensor=roofline_tensor, cqt=cq, train_step=train,
                    one_hour_sharded=hour, gpu_eager_baseline=eager, cpu_baseline=cpu, clocks=clocks)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


_RESULT_FD = None


def claim_stdout():
    """The contract is ONE JSON line on rank 0's stdout.  Libraries print there too (NCCL's version banner on process-group creation,
    for one): from here on file descriptor 1 is stderr for everything but emit()."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + '\n').encode()
    if _RESULT_FD is None:
        os.write(1, data)
    else:
        os.write(_RESULT_FD, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--blocks', type=int, default=256, help='3 s blocks per GPU per step')
    ap.add_argument('--no-early', action='store_true', help='end-to-end arm: copy the activations out only after the whole step')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-train', action='store_true', help='skip the loss-step leg (BASELINE.json configs[3])')
    ap.add_argument('--no-hour', action='store_true', help='skip the sharded one-hour-clip leg (BASELINE.json configs[4])')
    ap.add_argument('--no-eager', action='store_true', help='skip the eager-PyTorch GPU anchor')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the activations and audio of the last device-resident step as DIR/<name>.npy '
                         '(float32; larger outputs as a fixed, seeded sample, 48 MiB in all) on rank 0')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a CUDA device: timbre_trap_b200 has no CPU path')
    run_ours(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
