"""SURVEY section 8(f1): a Lightning checkpoint of the reference loads UNCHANGED into the engine's classes.

The evaluation driver does ``torch.load(run_dir/best.ckpt)['state_dict']`` and ``load_state_dict`` on a
LightningModule whose ``self.model`` is the network (the reference's src/ts_hear_test.py:18-34,
ts_hear_embed_pl_module.py:25), so every key carries a ``model.`` prefix; real asteroid registers one extra buffer
per filterbank (``torch_window``).  The checkpoints hold the state_dict of a seeded reference module: key names and
shapes as recorded from the reference (ckpt_keys.json), values as the seeded init reproduces them, checked against
the reference's own per-key fingerprint (ref_pins.npz; both written by tests/golden/make_golden.py).
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn as nn

from lookoncetohear_b200 import EmbedTFGridNet, Net, synth
from lookoncetohear_b200.net import SepState
from oracle import golden
from oracle import restate as rs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def pins():
    return np.load(os.path.join(GOLD, "ref_pins.npz"))


class _PLShaped(nn.Module):
    """What Lightning's state_dict looks like from outside: the network lives under ``self.model``."""

    def __init__(self, model):
        super().__init__()
        self.model = model


def _reference_state_dict(pins, name, seed, module):
    """The state_dict of the reference's `name` ('sep' / 'embed') network built under torch.manual_seed(seed)."""
    torch.manual_seed(seed)
    sd = {k: v.detach().clone() for k, v in module().state_dict().items()}
    with open(os.path.join(GOLD, "ckpt_keys.json")) as f:
        assert {k: list(v.shape) for k, v in sd.items()} == json.load(f)[name]
    assert golden.fingerprint_mismatches(pins, f"init_{name}_{seed}", sd) == []
    return sd


def _write_ckpt(path, net_sd, extra=None):
    sd = {"model." + k: v for k, v in net_sd.items()}                 # _PLShaped(network).state_dict()
    sd.update(extra or {})
    torch.save({"state_dict": sd, "epoch": 7, "global_step": 1234}, path)
    return sd


def test_separator_checkpoint_loads_strict(tmp_path, tsh_params, pins):
    ref = _reference_state_dict(pins, "sep", 11, lambda: Net(**tsh_params))
    path = os.path.join(tmp_path, "best.ckpt")
    extra = {"model.tfgridnet.enc.filterbank.torch_window": torch.hann_window(192),
             "model.tfgridnet.dec.filterbank.torch_window": torch.hann_window(192)}
    sd = _write_ckpt(path, ref, extra)
    torch.manual_seed(99)                                   # different init: everything must come from the file
    mine = _PLShaped(Net(**tsh_params))
    state = torch.load(path, map_location="cpu")["state_dict"]
    mine.load_state_dict(state, strict=True)                # ts_hear_test.py:23-26
    got = mine.state_dict()
    assert set(got) == set(sd) - set(extra)
    for k, v in got.items():
        assert torch.equal(v, sd[k]), k
    assert mine.model._dirty                                # the engine repacks on the next call


def test_enrollment_checkpoint_loads_strict(tmp_path, embed_params, pins):
    ref = _reference_state_dict(pins, "embed", 12, lambda: EmbedTFGridNet(**embed_params))
    path = os.path.join(tmp_path, "embed.ckpt")
    sd = _write_ckpt(path, ref)
    torch.manual_seed(98)
    mine = _PLShaped(EmbedTFGridNet(**embed_params))
    mine.load_state_dict(torch.load(path, map_location="cpu")["state_dict"], strict=True)
    for k, v in mine.state_dict().items():
        assert torch.equal(v, sd[k]), k
    assert any(k.startswith("model.blocks.0.attn_conv_Q_3.") for k in sd)      # espnet2 per-head naming


def test_state_dict_keys_match_reference_fixture(tsh_params, embed_params):
    """Key names / shapes of both networks == those of the reference modules (fixture made from the reference)."""
    with open(os.path.join(GOLD, "ckpt_keys.json")) as f:
        gold = json.load(f)
    for name, mod in (("sep", Net(**tsh_params)), ("embed", EmbedTFGridNet(**embed_params))):
        mine = {k: list(v.shape) for k, v in mod.state_dict().items()}
        assert mine == gold[name], name


def test_load_reference_state_roundtrip(tsh_params):
    """SepState.load_reference(reference-format dict).to_reference() is the identity (layout from the C ABI)."""
    torch.manual_seed(5)
    net = Net(**tsh_params)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    x, _ = synth.mixture(2, 128 * 53)
    e = synth.embedding(2)
    st = rs.sep_init_state(sd, 2)
    _, st = rs.sep_predict(sd, x, e[:, 0], st)
    hb, stride, offs = net._state_layout()
    buf = torch.zeros(hb // 4 + 2 * stride)
    back = SepState(buf, 2, 3, hb, stride, offs).load_reference(st).to_reference()
    for k in ("conv_buf", "deconv_buf", "istft_buf"):
        assert torch.equal(back[k], st[k]), k
    for i in range(3):
        for k in ("K_buf", "V_buf", "h0", "c0"):
            assert torch.equal(back["gridnet_bufs"][f"buf{i}"][k], st["gridnet_bufs"][f"buf{i}"][k]), (i, k)


def test_net_deepcopy_and_pickle(tsh_params):
    import copy
    import pickle
    net = Net(**tsh_params)
    net._engine()                                           # a live ctypes handle must not break copying
    for other in (copy.deepcopy(net), pickle.loads(pickle.dumps(net))):
        assert other._handle is None and other._dirty
        for (k, a), (_, b) in zip(net.state_dict().items(), other.state_dict().items()):
            assert torch.equal(a, b), k


@pytest.mark.gpu
def test_checkpoint_outputs_on_gpu(tmp_path, tsh_params, pins):
    ref = _reference_state_dict(pins, "sep", 13, lambda: Net(**tsh_params))
    path = os.path.join(tmp_path, "best.ckpt")
    _write_ckpt(path, ref)
    mine = _PLShaped(Net(**tsh_params))
    mine.load_state_dict(torch.load(path, map_location="cpu")["state_dict"], strict=True)
    mine = mine.eval().cuda()
    x, _ = synth.mixture(1, 128 * 12)
    e = synth.embedding(1)
    with torch.no_grad():
        y = mine.model(x.cuda(), e.cuda()).cpu()
    assert rs.rel_l2(y, torch.from_numpy(pins["ckpt_gpu.y"])) <= 1e-3


@pytest.mark.gpu
def test_stream_continues_from_reference_state(tsh_params):
    """A stream started on the reference implementation (here: the oracle, which produces the reference's state
    format) continues on the engine after SepState.load_reference()."""
    torch.manual_seed(3)
    net = Net(**tsh_params).eval()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    T0, T1 = 57, 9
    x, _ = synth.mixture(1, 128 * (T0 + T1))
    e = synth.embedding(1)
    xp = torch.nn.functional.pad(x, (0, 64))
    st = rs.sep_init_state(sd, 1)
    _, st = rs.sep_predict(sd, xp[..., :128 * T0 + 64], e[:, 0], st, pad=False)
    import copy
    y_ref, _ = rs.sep_predict(sd, xp[..., 128 * T0:], e[:, 0], copy.deepcopy(st), pad=False)
    net = net.cuda()
    gst = net.init_buffers(1, "cuda").load_reference(st)
    with torch.no_grad():
        y, _ = net.predict(xp[..., 128 * T0:].cuda(), e[:, 0].cuda(), gst, pad=False)
    assert rs.rel_l2(y.cpu(), y_ref) <= 1e-3
