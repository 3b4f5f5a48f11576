"""Pin the oracle (oracle/restate.py) against the reference: every comparison is with results of the
reference's own code, recorded in the committed fixtures by tests/golden/make_golden.py (ref_pins.npz
holds the large ones as samples plus norms, oracle/golden.py).  The reference repo has no golden
vectors of its own (SURVEY.md section 4)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from lookoncetohear_b200 import EmbedTFGridNet, Net, synth
from oracle import golden
from oracle import restate as rs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def pins():
    return np.load(os.path.join(GOLD, "ref_pins.npz"))


def _wsum(sd):
    return np.array([float(sum(v.double().abs().sum() for v in sd.values())),
                     float(sum((v.double() ** 2).sum() for v in sd.values()))])


def _seeded_sd(tsh_params, seed):
    torch.manual_seed(seed)
    return {k: v.detach().clone() for k, v in Net(**tsh_params).state_dict().items()}


def test_seeded_init_matches_reference(tsh_params, pins):
    """The engine's parameter containers under a seed hold the reference's seeded default init."""
    assert golden.fingerprint_mismatches(pins, "init_sep_0", _seeded_sd(tsh_params, 0), atol=1e-7) == []


def test_param_counts(pins, tsh_params, embed_params):
    for name, total, mod in (("sep", 2_037_960, Net(**tsh_params)), ("embed", 2_368_681, EmbedTFGridNet(**embed_params))):
        ref = dict(zip(pins[f"params_{name}.names"].tolist(), pins[f"params_{name}.numel"].tolist()))
        assert sum(ref.values()) == total, name
        assert {k: p.numel() for k, p in mod.named_parameters()} == ref, name


def test_restatement_equals_reference_forward_and_state(tsh_params, pins):
    sd = _seeded_sd(tsh_params, 3)
    assert np.allclose(_wsum(sd), pins["fwd_state.wsum"], rtol=1e-9), "seeded init differs from the build that made the fixture"
    x, _ = synth.mixture(2, 128 * 9 + 77, seed0=50)
    e = synth.embedding(2, seed0=60)
    st = rs.sep_init_state(sd, 2)
    y, st = rs.sep_predict(sd, x, e[:, 0], st)
    assert rs.rel_l2(y, torch.from_numpy(pins["fwd_state.y"])) < 5e-6
    for k in ("conv_buf", "deconv_buf", "istft_buf"):
        assert golden.pin_error(pins, f"fwd_state.{k}", st[k]) < 5e-6, k
    for i in range(3):
        for k in ("K_buf", "V_buf", "h0", "c0"):
            assert golden.pin_error(pins, f"fwd_state.buf{i}.{k}", st["gridnet_bufs"][f"buf{i}"][k]) < 5e-6, (i, k)


def test_restatement_fp64_floor(tsh_params, pins):
    sd = _seeded_sd(tsh_params, 1)
    assert np.allclose(_wsum(sd), pins["fp64_floor.wsum"], rtol=1e-9), "seeded init differs from the build that made the fixture"
    x, _ = synth.mixture(1, 128 * 8)
    e = synth.embedding(1)
    y64 = rs.sep_forward(rs.cast_sd(sd, torch.float64), x.double(), e.double())
    assert rs.rel_l2(y64, torch.from_numpy(pins["fp64_floor.y"])) < 5e-6


def test_embed_restatement_equals_reference(embed_params, pins):
    torch.manual_seed(2)
    sd = {k: v.detach().clone() for k, v in EmbedTFGridNet(**embed_params).state_dict().items()}
    assert np.allclose(_wsum(sd), pins["embed.wsum"], rtol=1e-9), "seeded init differs from the build that made the fixture"
    o = rs.embed_forward(sd, synth.enrollment(2, 5000))
    r = torch.from_numpy(pins["embed.emb"])
    assert rs.rel_l2(o, r) < 5e-5
    assert float(F.cosine_similarity(o, r).min()) > 0.99999


def test_restatement_streaming_equals_whole(tsh_params):
    sd = _seeded_sd(tsh_params, 5)
    x, _ = synth.mixture(1, 128 * 7)
    e = synth.embedding(1)
    y = rs.sep_forward(sd, x, e)
    st = rs.sep_init_state(sd, 1)
    xp = F.pad(x, (0, 64))
    ys = torch.cat([rs.sep_predict(sd, xp[..., 128 * i:128 * i + 192], e[:, 0], st, pad=False)[0]
                    for i in range(7)], -1)
    assert rs.rel_l2(ys, y) < 5e-6


def test_fast_timing_mode_equals_explicit_loop(tsh_params):
    sd = _seeded_sd(tsh_params, 6)
    x, _ = synth.mixture(1, 128 * 5)
    e = synth.embedding(1)
    y = rs.sep_forward(sd, x, e)
    rs.set_fast(True)
    try:
        yf = rs.sep_forward(sd, x, e)
    finally:
        rs.set_fast(False)
    assert rs.rel_l2(yf, y) < 5e-6


def test_golden_sep(tsh_params):
    g = np.load(os.path.join(GOLD, "sep_golden.npz"))
    sd = _seeded_sd(tsh_params, int(g["seed"]))
    assert np.allclose(_wsum(sd), g["wsum"], rtol=1e-9), "seeded init differs from the build that made the fixture"
    B, N = int(g["B"]), int(g["N"])
    x, _ = synth.mixture(B, N)
    e = synth.embedding(B)
    st = rs.sep_init_state(sd, B)
    y, st = rs.sep_predict(sd, x, e[:, 0], st)
    assert rs.rel_l2(y, torch.from_numpy(g["y"])) < 5e-6
    assert rs.rel_l2(st["gridnet_bufs"]["buf2"]["h0"], torch.from_numpy(g["h0_buf2"])) < 5e-6


def test_golden_embed(embed_params):
    g = np.load(os.path.join(GOLD, "embed_golden.npz"))
    from lookoncetohear_b200.embed import EmbedTFGridNet
    torch.manual_seed(int(g["seed"]))
    sd = {k: v.detach().clone() for k, v in EmbedTFGridNet(**embed_params).state_dict().items()}
    assert np.allclose(_wsum(sd), g["wsum"], rtol=1e-9)
    o = rs.embed_forward(sd, synth.enrollment(2, int(g["n"])))
    assert rs.rel_l2(o, torch.from_numpy(g["emb"])) < 5e-5


def test_si_sdr_known_answer():
    t = torch.sin(torch.arange(1000.) * 0.1)[None]
    n = torch.cos(torch.arange(1000.) * 0.37)[None]
    n = n - (n * t).sum() / (t * t).sum() * t          # orthogonal noise
    p = 3.0 * t + 0.3 * n * (t.norm() / n.norm()) * 3.0
    assert abs(float(rs.si_sdr(p, t)) - 20 * np.log10(1 / 0.3)) < 1e-3


def test_stft_shim_equals_the_stft_the_reference_vendors(pins, monkeypatch):
    """The one piece of espnet2 arithmetic the reference DOES carry -- Stft.forward, src/models/tfgridnet_orig/
    stft.py:68-195, identical to what espnet2's STFTEncoder calls -- pins the shim the enrollment oracle uses
    (oracle/shims/espnet2/enh/encoder/stft_encoder.py): same frames, same bins, same values, same output lengths."""
    monkeypatch.syspath_prepend(os.path.join(ROOT, "oracle", "shims"))
    from espnet2.enh.encoder.stft_encoder import STFTEncoder
    for j, (n_fft, hop, n) in enumerate(((128, 64, 5000), (128, 64, 4999), (192, 128, 3001))):
        x = synth.enrollment(3, n).transpose(1, 2).contiguous()          # [B, N, M] as EmbedTFGridNet.forward passes it
        ilens = torch.tensor([n, n, n])
        got, gl_out = STFTEncoder(n_fft, n_fft, hop, window="hann")(x, ilens)                             # complex [B,T,M,F]
        ref_shape = tuple(pins[f"stft{j}.shape"])                                                          # [B,T,M,F,2]
        assert got.shape == ref_shape[:-1] and got.shape[1] == 1 + n // hop
        assert gl_out.tolist() == pins[f"stft{j}.olens"].tolist()
        assert golden.pin_error(pins, f"stft{j}", torch.view_as_real(got)) < 1e-6
