"""Binaural cue errors on the GPU (l2h_eval_binaural, lookoncetohear_b200.metrics.binaural_errors / ild_diff / itd_diff)
against the reference's own results (tests/golden/binaural_golden.npz), the float64 restatement
(tests/binaural_oracle.py) and known answers rendered with the engine's own renderer."""
import ctypes

import numpy as np
import pytest
import torch

import binaural_oracle as bo
from lookoncetohear_b200 import Net, _cabi, synth
from lookoncetohear_b200.metrics import binaural_errors, ild_diff, itd_diff
from lookoncetohear_b200.render import render_binaural
from test_binaural_cpu import CASES, GOLDEN, assert_same_nonfinite_and_close, check_lags, tied_mixtures

pytestmark = pytest.mark.gpu


def lags_of(itd_us, sr):
    return torch.round(itd_us.double() * sr / 1e6).long()


def assert_itd_is_mean_of_own_windows(out, win):
    """moving: itd_diff = mean over valid windows of |itd_est - itd_gt|, from the same call's per-window values."""
    win = win.cpu().double()
    v = win[..., 4] != 0
    d = (win[..., 2] - win[..., 3]).abs()
    want = torch.stack([d[b][v[b]].mean() for b in range(d.shape[0])])
    assert_same_nonfinite_and_close(out[:, 1].cpu(), want, 1e-3)


def check_against_restatement(e, g, sr, moving, out, win):
    """e, g: the CPU inputs; out [B, 2], win [B, C, 5] from the GPU."""
    w = bo.binaural_windows(e, g, sr, moving)
    out, win = out.cpu().double(), win.cpu().double()
    assert torch.equal(win[..., 4] != 0, w["valid"])
    near_tie = torch.zeros_like(w["valid"])
    for i, tag in ((0, "est"), (1, "gt")):
        assert_same_nonfinite_and_close(win[..., i], w[f"ild_{tag}"], 1e-4)
        c = w[f"corr_{tag}"].abs()
        tau = lags_of(win[..., 2 + i], sr)
        assert (tau.abs() <= w["t"]).all()
        picked = c.gather(-1, (tau + w["t"])[..., None])[..., 0]
        best = c.amax(-1)
        # the correlation behind the chosen lag is the largest up to 1e-6 ||l|| ||r||
        assert (best - picked <= 1e-6 * w[f"norm_{tag}"] + 1e-30).all(), (best - picked).max()
        top2 = c.topk(2, dim=-1).values
        near_tie |= (top2[..., 0] - top2[..., 1]) < 1e-5 * w[f"norm_{tag}"]
    assert_same_nonfinite_and_close(out[:, 0], bo.ild_diff(e, g, sr, moving), 1e-4)
    assert_itd_is_mean_of_own_windows(out, win)
    clear = ~near_tie.any(1)
    assert_same_nonfinite_and_close(out[clear, 1], bo.itd_diff(e, g, sr, moving)[clear], 1e-3)


@pytest.mark.parametrize("moving", [False, True], ids=["static", "moving"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_matches_reference_fixture(name, moving):
    sr, e, g = CASES[name]
    key = f"{name}.{'moving' if moving else 'static'}"
    out, win = binaural_errors(torch.from_numpy(e).cuda(), torch.from_numpy(g).cuda(), sr, moving, return_windows=True)
    winc = win.cpu().double().numpy()
    assert np.array_equal(winc[..., 4] != 0, GOLDEN[key + ".valid"])
    for i, tag in ((0, "est"), (1, "gt")):
        assert_same_nonfinite_and_close(winc[..., i], GOLDEN[f"{key}.ild_{tag}"], 1e-4)
        check_lags(lags_of(win[..., 2 + i].cpu(), sr).numpy(), key, tag)
    outc = out.cpu().double().numpy()
    assert_same_nonfinite_and_close(outc[:, 0], GOLDEN[key + ".ild_diff"], 1e-4)
    ok = ~tied_mixtures(key)
    assert_same_nonfinite_and_close(outc[ok, 1], GOLDEN[key + ".itd_diff"][ok], 1e-3)
    if moving:
        assert_itd_is_mean_of_own_windows(out, win)
    # the drop-ins return the same columns
    ge, gg = torch.from_numpy(e).cuda(), torch.from_numpy(g).cuda()
    assert_same_nonfinite_and_close(ild_diff(ge, gg, sr, moving).cpu(), outc[:, 0], 1e-5)
    torch.testing.assert_close(itd_diff(ge, gg, sr, moving).cpu(), out[:, 1].cpu(), rtol=0, atol=0, equal_nan=True)
    if not moving:                                               # static ILD needs no sampling rate
        assert_same_nonfinite_and_close(ild_diff(ge, gg).cpu(), outc[:, 0], 1e-5)


@pytest.mark.parametrize("moving", [False, True], ids=["static", "moving"])
@pytest.mark.parametrize("B,T,sr", [(1, 1002, 8000), (3, 64000, 16000), (64, 80000, 16000), (3, 80000, 48000),
                                    (1, 64000, 48000), (64, 1002, 8000), (3, 1002, 48000)])
def test_gpu_matches_restatement(B, T, sr, moving):
    rng = np.random.RandomState(B * 7 + T + sr)
    e, g = bo._speechlike(rng, B, T, sr)
    if B > 1:                                                    # one mixture of independent noise: no true lag
        e[-1], g[-1] = 0.05 * rng.randn(2, T), 0.05 * rng.randn(2, T)
    e, g = torch.from_numpy(e).float(), torch.from_numpy(g).float()
    out, win = binaural_errors(e.cuda(), g.cuda(), sr, moving, return_windows=True)
    check_against_restatement(e, g, sr, moving, out, win)


@pytest.mark.parametrize("moving", [False, True], ids=["static", "moving"])
def test_known_cues_through_the_renderer(moving):
    """left = delta[n - d_l] * src, right = g delta[n - d_r] * src of a noise source that is zero for 64 samples around
    every 250 ms boundary: in every window the pair's ITD is (d_l - d_r) / sr * 1e6 exactly and its ILD -20 log10 g."""
    sr, N = 16000, 64000
    gen = torch.Generator().manual_seed(3)
    src = 0.1 * torch.randn(1, 1, N, generator=gen)
    for k in range(0, N + 1, 4000):
        src[..., max(k - 64, 0):k + 64] = 0

    def render(d_l, d_r, gain):
        rir = torch.zeros(1, 1, 2, 64)
        rir[0, 0, 0, d_l] = 1.0
        rir[0, 0, 1, d_r] = gain
        ev, _, norm = render_binaural(src.cuda(), rir.cuda())
        assert float(norm[0]) == 1.0
        return ev[:, 0]

    gt, est = render(3, 12, 0.5), render(20, 7, 1.25)            # ITD -562.5 us / +812.5 us
    got = binaural_errors(est, gt, sr, moving).cpu().double()
    want_itd = abs((20 - 7) / sr * 1e6 - (3 - 12) / sr * 1e6)
    want_ild = abs(-20 * np.log10(1.25) + 20 * np.log10(0.5))
    assert abs(float(got[0, 1]) - want_itd) < (1e-3 if moving else 1e-9), got
    assert abs(float(got[0, 0]) - want_ild) < 1e-4, got
    assert float(itd_diff(est, gt, sr, moving)[0]) == float(got[0, 1])


def test_refusals():
    x = torch.randn(2, 2, 64001, device="cuda")
    with pytest.raises(RuntimeError, match="even window length"):
        itd_diff(x, x, 16000)                                    # static, odd T
    y = torch.randn(2, 2, 88200, device="cuda")
    with pytest.raises(RuntimeError, match="even window length, got 11025"):
        binaural_errors(y, y, 44100, moving=True)                # FW = 11025
    assert torch.isfinite(ild_diff(x, x)).all()                  # ILD alone: any length
    assert torch.isfinite(ild_diff(y, y, 44100, moving=True)).all()
    z = torch.randn(1, 2, 2000, device="cuda")
    with pytest.raises(RuntimeError, match="exceeds 256"):
        binaural_errors(z, z, 300000)                            # TMAX = 300
    n = ctypes.c_size_t()
    assert _cabi.lib().l2h_eval_binaural_workspace_bytes(1, 2000, 0, 257, ctypes.byref(n)) != 0
    assert _cabi.lib().l2h_eval_binaural_workspace_bytes(1, 2000, 0, 256, ctypes.byref(n)) == 0


def test_two_calls_are_bit_identical():
    rng = np.random.RandomState(9)
    e, g = bo._speechlike(rng, 16, 64000, 16000)
    e, g = torch.from_numpy(e).float().cuda(), torch.from_numpy(g).float().cuda()
    for moving in (False, True):
        a = binaural_errors(e, g, 16000, moving, return_windows=True)
        b = binaural_errors(e, g, 16000, moving, return_windows=True)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def test_separator_output_end_to_end(tsh_params):
    """Net output -> binaural_errors without the audio leaving the device; checked on the copied-back output."""
    torch.manual_seed(0)
    net = Net(**tsh_params).eval().cuda()
    mix, tgt = synth.mixture(2, 128 * 64)
    e = synth.embedding(2)
    with torch.no_grad():
        y = net(mix.cuda(), e.cuda())
    g = tgt.cuda()
    for moving in (False, True):
        out, win = binaural_errors(y, g, 16000, moving, return_windows=True)
        assert out.is_cuda and out.shape == (2, 2)
        check_against_restatement(y.cpu(), tgt, 16000, moving, out, win)


def test_eval_batch_256_moving():
    """B = 256 x 4 s at 16 kHz, moving; a sample of the mixtures against the restatement."""
    rng = np.random.RandomState(256)
    e, g = bo._speechlike(rng, 256, 64000, 16000)
    e, g = torch.from_numpy(e).float(), torch.from_numpy(g).float()
    out, win = binaural_errors(e.cuda(), g.cuda(), 16000, True, return_windows=True)
    idx = torch.tensor([0, 1, 77, 128, 200, 255])
    check_against_restatement(e[idx], g[idx], 16000, True, out[idx], win[idx])
