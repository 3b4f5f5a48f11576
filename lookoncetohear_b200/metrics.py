"""Evaluation epilogue on the GPU: the per-mixture figures of the reference's evaluation loop
(src/ts_hear_test.py:139-146 -- SI-SNR of the output, SI-SNR improvement over the mixture, cosine similarity of
the enrollment embedding) computed from the separator's DEVICE output by ``l2h_eval_metrics``; only three floats
per mixture cross to the host.  The binaural cue errors of src/eval/binaural.py (ILD / ITD, static and moving-source)
come from ``l2h_eval_binaural`` in one pass.  No CPU fallback."""
import ctypes

import torch

from . import _cabi


def eval_metrics(outputs, target, mixture=None, embedding=None, embedding_gt=None):
    """outputs / target / mixture: [B, C, N] CUDA tensors; embedding / embedding_gt: [B, D] or [B, 1, D].
    Returns a [B, 3] CUDA tensor: (output_sisnr, si_snr_i, embedding_sim)."""
    if not outputs.is_cuda:
        raise RuntimeError("lookoncetohear_b200.metrics.eval_metrics needs CUDA tensors (no CPU fallback)")
    dev = outputs.device
    est = outputs.contiguous().float()
    tgt = target.to(dev, torch.float32).contiguous()
    if tgt.shape != est.shape:
        raise ValueError(f"target shape {tuple(tgt.shape)} != output shape {tuple(est.shape)}")
    mix = mixture.to(dev, torch.float32).contiguous() if mixture is not None else None
    B, C, N = est.shape
    emb = emb_gt = None
    D = 0
    if embedding is not None and embedding_gt is not None:
        emb = embedding.to(dev, torch.float32).reshape(B, -1).contiguous()
        emb_gt = embedding_gt.to(dev, torch.float32).reshape(B, -1).contiguous()
        D = emb.shape[1]
    out = torch.empty(B, 3, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(_cabi.lib().l2h_eval_metrics(
            est.data_ptr(), tgt.data_ptr(), mix.data_ptr() if mix is not None else None, B, C, N,
            emb.data_ptr() if emb is not None else None, emb_gt.data_ptr() if emb_gt is not None else None, D,
            out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
    return out


# ----------------------------------------------------------------------------- binaural cues (src/eval/binaural.py)

RMS_THRESHOLD = 1e-3          # chunk_and_mask's rms_threshold (binaural.py:7)


def frame_width(sr):
    """The moving-source window in samples, FW = int(round(1e-3 * 250 * sr)) (binaural.py:19); Python rounds half
    to even, e.g. 22050 Hz -> 5512."""
    return int(round(1e-3 * 250 * sr))


def max_lag(sr):
    """TMAX = int(round(1e-3 * sr)) (binaural.py:125), the largest lag the ITD search considers."""
    return int(round(1e-3 * sr))


def _binaural(s_est, s_gt, sr, moving, t_max, return_windows):
    if s_est.dim() != 3 or s_est.shape[1] != 2 or s_est.shape[2] < 1 or tuple(s_gt.shape) != tuple(s_est.shape):
        raise ValueError(f"s_est and s_gt must both be [B, 2, T] (ear 0 = left), got {tuple(s_est.shape)} and "
                         f"{tuple(s_gt.shape)}")
    if not (s_est.is_cuda and s_gt.is_cuda):
        raise RuntimeError("lookoncetohear_b200.metrics binaural cues need CUDA tensors (no CPU fallback)")
    if moving and sr is None:
        raise ValueError("moving=True needs sr to size the 250 ms windows")
    dev = s_est.device
    est = s_est.to(dev, torch.float32).contiguous()
    gt = s_gt.to(dev, torch.float32).contiguous()
    B, _, T = est.shape
    frame = frame_width(sr) if moving else 0
    if moving and frame < 1:
        raise ValueError(f"sr = {sr} gives an empty 250 ms window")
    n_win = 1 + (T - 1) // frame if moving else 1
    lib = _cabi.lib()
    nbytes = ctypes.c_size_t()
    _cabi.check(lib.l2h_eval_binaural_workspace_bytes(B, T, frame, t_max, ctypes.byref(nbytes)))
    out = torch.empty(B, 2, dtype=torch.float32, device=dev)
    win = torch.empty(B, n_win, 5, dtype=torch.float32, device=dev) if return_windows else None
    ws = torch.empty(max(int(nbytes.value), 8), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _cabi.check(lib.l2h_eval_binaural(
            est.data_ptr(), gt.data_ptr(), B, T, frame, t_max, RMS_THRESHOLD, int(sr) if sr else 0, out.data_ptr(),
            win.data_ptr() if win is not None else None, ws.data_ptr(), ws.numel(),
            torch.cuda.current_stream(dev).cuda_stream))
    return (out, win) if return_windows else out


def binaural_errors(s_est, s_gt, sr, moving=False, return_windows=False):
    """ILD and ITD errors of one pass.  s_est / s_gt: [B, 2, T] CUDA tensors (ear 0 = left), sr in Hz.
    Returns a [B, 2] CUDA tensor (ild_diff dB, itd_diff us) -- binaural.py's ild_diff / itd_diff -- and with
    return_windows also the per-window [B, n_windows, 5] tensor (ild_est, ild_gt, itd_est, itd_gt, valid).
    The window length (T, or the 250 ms frame when moving) must be even: the reference's ITD is undefined otherwise."""
    t_max = max_lag(sr)
    if t_max < 1:
        raise ValueError(f"sr = {sr} gives TMAX = 0: no lag to search")
    return _binaural(s_est, s_gt, sr, moving, t_max, return_windows)


def ild_diff(s_est, s_gt, sr=None, moving=False):
    """binaural.py:49-81 on the GPU: [B] CUDA tensor of ILD errors in dB.  sr is needed only when moving.
    Any signal length works (no lag search)."""
    return _binaural(s_est, s_gt, sr, moving, 0, False)[:, 0]


def itd_diff(s_est, s_gt, sr, moving=False):
    """binaural.py:120-149 on the GPU: [B] CUDA tensor of ITD errors in microseconds."""
    return binaural_errors(s_est, s_gt, sr, moving)[:, 1]
