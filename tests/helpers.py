import numpy as np
import torch


def tonal_clip(n_samples, sample_rate, seed, n_batch=1):
    """Same generator as scripts/make_golden.py (harmonic tones + -30 dB noise, peak-normalised)."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_samples) / sample_rate
    out = []
    for _ in range(n_batch):
        x = np.zeros(n_samples)
        for midi in rng.integers(40, 90, size=4):
            f0 = 440.0 * 2 ** ((midi - 69) / 12)
            for h in range(1, 5):
                if f0 * h < 0.45 * sample_rate:
                    x += np.sin(2 * np.pi * f0 * h * t + rng.uniform(0, 2 * np.pi)) / h
        x += 10 ** (-30 / 20) * rng.standard_normal(n_samples)
        out.append(x / np.abs(x).max())
    return torch.from_numpy(np.stack(out)[:, None, :].astype(np.float32))


def rel_err(a, b):
    """(max-abs error / max|b|, l2 error / ||b||) - the norm-relative bounds of SURVEY.md section 8c."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)), float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def check_step_gradients(got, want, tag, floorless=None):
    """Each parameter: err <= 0.1 |g| + 0.01 |g_total| (the floor for the tiny bias vectors, whose bf16 noise does not shrink with
    them), and the global gradient at rel-L2 <= 3e-2.  `floorless`: also err <= floorless * |g| WITHOUT the floor for every parameter
    whose gradient norm is at least 1e-3 of the total - the floor would let a wrong small layer, bias or skip weight through."""
    assert set(got) == set(want)
    total_norm = sum(float(v.norm()) ** 2 for v in want.values()) ** 0.5
    num = den = 0.0
    worst = worst_gated = (0.0, None)
    failed = []
    for k in want:
        assert got[k].shape == want[k].shape, k
        err, ref = float((got[k] - want[k]).norm()), float(want[k].norm())
        num += err ** 2
        den += ref ** 2
        rel = err / max(ref, 1e-12)
        if rel > worst[0]:
            worst = (rel, k)
        if err > 1e-1 * ref + 1e-2 * total_norm:
            failed.append((k, err, ref, total_norm))
        if floorless is not None and ref >= 1e-3 * total_norm:
            if rel > worst_gated[0]:
                worst_gated = (rel, k)
            if rel > floorless:
                failed.append((k, 'floorless', rel, ref / total_norm))
    print(f'{tag}: global gradient rel-L2 error', (num / den) ** 0.5, 'worst parameter', worst, 'worst of the floorless gate', worst_gated)
    assert not failed, failed
    assert (num / den) ** 0.5 <= 3e-2, ((num / den) ** 0.5, worst)


def tonal_clip_with_pitches(n_samples, sample_rate, seed):
    """As tonal_clip (one item) but also returns the MIDI pitches of the four fundamentals."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_samples) / sample_rate
    x = np.zeros(n_samples)
    midis = rng.integers(40, 90, size=4)
    for midi in midis:
        f0 = 440.0 * 2 ** ((midi - 69) / 12)
        for h in range(1, 5):
            if f0 * h < 0.45 * sample_rate:
                x += np.sin(2 * np.pi * f0 * h * t + rng.uniform(0, 2 * np.pi)) / h
    x += 10 ** (-30 / 20) * rng.standard_normal(n_samples)
    return torch.from_numpy((x / np.abs(x).max())[None, None, :].astype(np.float32)), midis


def pick_peaks(activations, t):
    """
    Restates the reference's evaluation post-processing (timbre_trap/utils/processing.py:66-124 via
    PitchDataset.activations_to_multi_pitch, PitchDataset.py:309-349, peaks_only=True): keep strict local maxima along the
    frequency axis (zero-padded edges, scipy.signal.argrelmax semantics), then binarise with `>= t`.  (F, T) -> bool (F, T).
    """
    a = np.asarray(activations, dtype=np.float64)
    p = np.pad(a, ((1, 1), (0, 0)))
    peaks = (p[1:-1] > p[:-2]) & (p[1:-1] > p[2:])
    return peaks & (a >= t)


def multipitch_prf(est, ref, tol_bins):
    """
    Frame-wise multi-pitch precision / recall / F1 in the manner of mir_eval.multipitch (matching within a pitch tolerance,
    here expressed in bins), est / ref: bool (F, T).  In one dimension the greedy left-to-right matching is a maximum matching.
    """
    tp = 0
    for e, r in zip(est.T, ref.T):
        ei, ri = np.flatnonzero(e), np.flatnonzero(r)
        i = j = 0
        while i < len(ei) and j < len(ri):
            if abs(int(ei[i]) - int(ri[j])) <= tol_bins:
                tp += 1; i += 1; j += 1
            elif ei[i] < ri[j]:
                i += 1
            else:
                j += 1
    n_est, n_ref = int(est.sum()), int(ref.sum())
    eps = np.finfo(float).eps
    p, r = tp / (n_est + eps), tp / (n_ref + eps)
    return p, r, 2 * p * r / (p + r + eps)
