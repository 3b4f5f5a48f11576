"""ORACLE for the binaural cue errors (test infrastructure; never imported by the product path).

A CPU restatement of src/eval/binaural.py:6-149 written from its formulas in float64 torch, with the cross-correlation as
direct circular lag sums instead of the reference's rfft / irfft, so that it shares no method with the code it checks:
    windows   static: one window of the whole signal; moving: FW = round(0.25 sr) samples, C = 1 + (T-1)//FW,
              zero padding past T, valid = max over ears of sqrt(mean(gt^2)) >= 1e-3            (chunk_and_mask :6-42)
    ILD       10 log10(sum l^2 / sum r^2)                                                         (compute_ild :44-47)
    ITD       tau / sr * 1e6, tau = first argmax over k in [-t, t] of |sum_n l[(n+k) mod L] r[n]|,
              t = min(round(1e-3 sr), L//2)                                        (axiswise_xcorr :83-92, compute_itd :94-117)
    per mixture  static |est - gt|; moving: ILD |mean_valid est - mean_valid gt|, ITD mean_valid |est - gt|
                                                                                   (ild_diff :49-81, itd_diff :120-149)
It is pinned to the reference's own results in tests/golden/binaural_golden.npz (tests/test_binaural_cpu.py); the inputs
of those results are regenerated here from seeds (``cases()``).
"""
import numpy as np
import torch


def frame_tmax(sr):
    """(FW, TMAX) with Python's rounding, as binaural.py:19 and :125 compute them."""
    return int(round(1e-3 * 250 * sr)), int(round(1e-3 * sr))


def _windows(x, L):
    """[B, 2, T] -> [B, 2, C, L], zero-padded at the end."""
    B, _, T = x.shape
    C = 1 + (T - 1) // L
    return torch.nn.functional.pad(x, (0, C * L - T)).reshape(B, 2, C, L)


def circular_xcorr(l, r, t):
    """c[..., k + t] = sum_n l[..., (n + k) mod L] * r[..., n] for k = -t .. t (direct lag sums, float64)."""
    return torch.stack([(torch.roll(l, -k, dims=-1) * r).sum(-1) for k in range(-t, t + 1)], dim=-1)


def binaural_windows(s_est, s_gt, sr=None, moving=False, with_itd=True):
    """Per-window cues.  Returns a dict of [B, C] tensors ild_est, ild_gt, tau_est, tau_gt (lag in samples), itd_est,
    itd_gt (us), valid (bool), and [B, C, 2t+1] corr_est / corr_gt, norm_est / norm_gt (= ||l|| ||r|| per window), t."""
    est, gt = torch.as_tensor(s_est).double(), torch.as_tensor(s_gt).double()
    T = est.shape[-1]
    if moving:
        FW, TMAX = frame_tmax(sr)
        L = FW
    else:
        L = T
        TMAX = frame_tmax(sr)[1] if sr is not None else 0
    we, wg = _windows(est, L), _windows(gt, L)                      # [B, 2, C, L]
    out = {}
    for tag, w in (("est", we), ("gt", wg)):
        el, er = (w[:, 0] ** 2).sum(-1), (w[:, 1] ** 2).sum(-1)
        out["ild_" + tag] = 10 * torch.log10(el / er)
        out["norm_" + tag] = el.sqrt() * er.sqrt()
    if moving:
        out["valid"] = (wg ** 2).mean(-1).sqrt().amax(1) >= 1e-3
    else:
        out["valid"] = torch.ones(est.shape[0], 1, dtype=torch.bool)
    if with_itd:
        if L % 2:
            raise ValueError(f"ITD needs an even window length, got {L}")
        t = min(TMAX, L // 2)
        out["t"] = t
        for tag, w in (("est", we), ("gt", wg)):
            c = circular_xcorr(w[:, 0], w[:, 1], t)
            tau = c.abs().argmax(-1) - t                              # torch.argmax: first maximum, as np.argmax
            out["corr_" + tag] = c
            out["tau_" + tag] = tau
            out["itd_" + tag] = tau.double() / sr * 1e6
    return out


def _masked_mean(v, m):
    return torch.stack([v[b][m[b]].mean() for b in range(v.shape[0])])   # empty -> NaN, as np.mean([])


def ild_diff(s_est, s_gt, sr=None, moving=False):
    w = binaural_windows(s_est, s_gt, sr, moving, with_itd=False)
    return (_masked_mean(w["ild_est"], w["valid"]) - _masked_mean(w["ild_gt"], w["valid"])).abs()


def itd_diff(s_est, s_gt, sr, moving=False):
    w = binaural_windows(s_est, s_gt, sr, moving)
    return _masked_mean((w["itd_est"] - w["itd_gt"]).abs(), w["valid"])


# ----------------------------------------------------------------------------- seeded inputs of the fixture


def _delayed_pair(src, d_l, d_r, g):
    """left = src delayed by d_l, right = g * src delayed by d_r (non-circular, zeros shifted in)."""
    T = src.shape[-1]
    out = np.zeros((2, T))
    out[0, d_l:] = src[:T - d_l]
    out[1, d_r:] = g * src[:T - d_r]
    return out


def _chirp_case():
    """The reference's own test (binaural.py:151-198): 8 kHz, 5 s chirps, right ear = left rolled by -shift and
    scaled by 0.5, shifts -4..4, estimate = gt + 0.1 N(0, 1)."""
    sr, dur = 8000, 5
    rng = np.random.RandomState(0)
    t = np.arange(0, dur, 1 / sr)
    x = np.cos(2 * np.pi * (100 + 250 * t) * t)
    gts, ests = [], []
    for shift in range(-4, 5):
        gt = np.stack([x, np.roll(x, -shift) * 0.5]) * 0.1
        ests.append(gt + rng.normal(0, 1, size=gt.shape) * 0.1)
        gts.append(gt)
    return sr, np.array(ests), np.array(gts)


def _speechlike(rng, B, T, sr):
    """Band-limited noise bursts with random per-mixture delays and gains; est = gt with other cues plus noise."""
    ests, gts = [], []
    tmax = int(round(1e-3 * sr))
    for _ in range(B):
        src = np.convolve(rng.randn(T + 64), np.hanning(9), mode="same")[:T]
        env = 0.5 + 0.5 * np.sin(2 * np.pi * rng.uniform(1, 4) * np.arange(T) / sr + rng.uniform(0, 6.3))
        src = 0.05 * src * env
        d = rng.randint(0, tmax + 1, size=4)
        g = rng.uniform(0.3, 1.5, size=2)
        gts.append(_delayed_pair(src, d[0], d[1], g[0]))
        ests.append(_delayed_pair(src, d[2], d[3], g[1]) + 0.01 * rng.randn(2, T))
    return np.array(ests), np.array(gts)


def cases():
    """name -> (sr, est [B, 2, T] float32, gt float32).  Everything from fixed seeds (numpy RandomState is stable)."""
    out = {}
    sr, e, g = _chirp_case()
    out["chirp8k"] = (sr, e, g)
    rng = np.random.RandomState(1)
    out["sr16k_64000"] = (16000,) + _speechlike(rng, 4, 64000, 16000)
    out["sr16k_65234"] = (16000,) + _speechlike(rng, 4, 65234, 16000)
    # windows silenced by zeroed 0.5 s stretches of gt (not aligned to the 250 ms frames); mixture 1: silent gt;
    # mixture 2: the estimate's right ear is silent; mixture 3: noise only, independent ears (no true lag, near-ties)
    e, g = _speechlike(rng, 4, 64000, 16000)
    g[0, :, 6000:14000] = 0
    g[0, :, 40000:48000] = 0
    g[1] = 0
    e[2, 1] = 0
    e[3] = 0.05 * rng.randn(2, 64000)
    g[3] = 0.05 * rng.randn(2, 64000)
    out["sr16k_edge"] = (16000, e, g)
    out["sr48k_1p5s"] = (48000,) + _speechlike(rng, 3, 72000, 48000)
    return {k: (sr, e.astype(np.float32), g.astype(np.float32)) for k, (sr, e, g) in out.items()}


def checksum(x):
    x = np.asarray(x, dtype=np.float64)
    return np.array([np.abs(x).sum(), (x ** 2).sum()])
