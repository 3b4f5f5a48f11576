"""The binaural cue restatement (tests/binaural_oracle.py) against the reference's own results
(tests/golden/binaural_golden.npz, written by tests/golden/make_binaural_golden.py from src/eval/binaural.py), and the
argument checks of the GPU wrappers, which run before any device is touched."""
import os

import numpy as np
import pytest
import torch

import binaural_oracle as bo

GOLDEN = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "binaural_golden.npz"))
CASES = bo.cases()
NEAR_TIE = 1e-5          # margin of the best |c| over the second, relative to ||l|| ||r||


def assert_same_nonfinite_and_close(got, want, atol):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want)), (got, want)
    assert np.array_equal(np.isposinf(got), np.isposinf(want)) and np.array_equal(np.isneginf(got), np.isneginf(want))
    fin = np.isfinite(want)
    assert np.allclose(got[fin], want[fin], rtol=0, atol=atol), np.abs(got[fin] - want[fin]).max()


def check_lags(tau, key, tag):
    """tau [B, C]: equal to the reference's lag where its margin is clear, else one of its two best lags."""
    tau = np.asarray(tau)
    margin, top2 = GOLDEN[f"{key}.margin_{tag}"], GOLDEN[f"{key}.top2_{tag}"]
    clear = margin >= NEAR_TIE
    assert np.array_equal(tau[clear], GOLDEN[f"{key}.tau_{tag}"][clear]), key
    assert ((tau[:, :, None] == top2).any(-1) | clear).all(), key


def tied_mixtures(key):
    return ((GOLDEN[f"{key}.margin_est"] < NEAR_TIE) | (GOLDEN[f"{key}.margin_gt"] < NEAR_TIE)).any(1)


def test_inputs_regenerate():
    assert sorted(CASES) == list(GOLDEN["cases"])
    for name, (sr, e, g) in CASES.items():
        assert int(GOLDEN[f"{name}.sr"]) == sr
        assert np.allclose(bo.checksum(e), GOLDEN[f"{name}.est_sum"], rtol=1e-12)
        assert np.allclose(bo.checksum(g), GOLDEN[f"{name}.gt_sum"], rtol=1e-12)


@pytest.mark.parametrize("moving", [False, True], ids=["static", "moving"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_matches_reference(name, moving):
    sr, e, g = CASES[name]
    key = f"{name}.{'moving' if moving else 'static'}"
    w = bo.binaural_windows(e, g, sr, moving)
    assert np.array_equal(w["valid"].numpy(), GOLDEN[key + ".valid"])
    for tag in ("est", "gt"):
        assert_same_nonfinite_and_close(w[f"ild_{tag}"], GOLDEN[f"{key}.ild_{tag}"], 1e-4)
        check_lags(w[f"tau_{tag}"].numpy(), key, tag)
    assert_same_nonfinite_and_close(bo.ild_diff(e, g, sr, moving), GOLDEN[key + ".ild_diff"], 1e-4)
    itd = bo.itd_diff(e, g, sr, moving).numpy()
    ok = ~tied_mixtures(key)
    assert ok.any()
    assert_same_nonfinite_and_close(itd[ok], GOLDEN[key + ".itd_diff"][ok], 1e-6)


def test_fixture_covers_the_edge_cases():
    """silent gt -> NaN ILD (and NaN moving ITD: no valid window); silent estimate ear -> inf ILD; silenced stretches
    -> invalid windows; all-zero correlations (silent ears) -> exact ties, resolved to the first lag -t."""
    assert np.isnan(GOLDEN["sr16k_edge.static.ild_diff"][1]) and np.isnan(GOLDEN["sr16k_edge.moving.itd_diff"][1])
    assert np.isposinf(GOLDEN["sr16k_edge.static.ild_diff"][2])
    assert not GOLDEN["sr16k_edge.moving.valid"][0].all() and GOLDEN["sr16k_edge.moving.valid"][0].any()
    assert tied_mixtures("sr16k_edge.moving")[1] and (GOLDEN["sr16k_edge.moving.tau_gt"][1] == -16).all()
    assert (GOLDEN["sr16k_edge.static.tau_est"][2] == -16).all()
    assert GOLDEN["sr16k_65234.moving.valid"].shape == (4, 17)
    assert int(GOLDEN["sr48k_1p5s.sr"]) == 48000


def test_frame_and_lag_rounding():
    from lookoncetohear_b200.metrics import frame_width, max_lag
    assert (frame_width(22050), max_lag(22050)) == (5512, 22) == bo.frame_tmax(22050)
    assert (frame_width(44100), max_lag(44100)) == (11025, 44)
    assert (frame_width(16000), max_lag(16000)) == (4000, 16)


def test_wrappers_refuse_cpu_tensors_and_bad_shapes():
    from lookoncetohear_b200.metrics import binaural_errors, ild_diff, itd_diff
    x = torch.zeros(2, 2, 1000)
    with pytest.raises(RuntimeError, match="CUDA"):
        binaural_errors(x, x, 16000)
    with pytest.raises(RuntimeError, match="CUDA"):
        ild_diff(x, x)
    with pytest.raises(RuntimeError, match="CUDA"):
        itd_diff(x, x, 16000, moving=True)
    for bad in (torch.zeros(2, 1000), torch.zeros(2, 3, 1000), torch.zeros(1, 2, 2, 1000)):
        with pytest.raises(ValueError):
            binaural_errors(bad, bad, 16000)
        with pytest.raises(ValueError):
            ild_diff(bad, bad)
    with pytest.raises(ValueError):
        itd_diff(x, torch.zeros(2, 2, 999), 16000)
