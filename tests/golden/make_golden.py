"""Generate the committed fixtures from the REFERENCE ITSELF (run where a checkout of the reference
exists, see oracle/ref_loader.py):  python tests/golden/make_golden.py

Weights are not stored (8 MB): they are the PyTorch default init under torch.manual_seed(seed),
which the reference modules and the engine's parameter containers reproduce identically
(tests/test_oracle.py::test_seeded_init_matches_reference); a checksum of the weights is stored
so that an RNG drift between torch builds is detected rather than misread as a parity failure.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lookoncetohear_b200 import synth  # noqa: E402
from oracle import golden  # noqa: E402
from oracle import ref_loader as rl  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def weight_checksum(sd):
    return np.array([float(sum(v.double().abs().sum() for v in sd.values())),
                     float(sum((v.double() ** 2).sum() for v in sd.values()))])


def main():
    torch.set_num_threads(8)
    # ---- separation: whole utterance (ragged length) + chunked streaming, B=2 ----------------
    seed = 0
    net = rl.reference_net(seed)
    B, N = 2, 128 * 14 - 51
    x, tgt = synth.mixture(B, N)
    e = synth.embedding(B)
    with torch.no_grad():
        y = net(x, e)
        st = net.init_buffers(B, "cpu")
        xp = torch.nn.functional.pad(x, (0, 128 * 14 - N + 64))
        ys = torch.cat([net.predict(xp[..., 128 * i:128 * i + 192], e[:, 0], st, pad=False)[0] for i in range(14)], -1)
    np.savez_compressed(os.path.join(HERE, "sep_golden.npz"), seed=seed, B=B, N=N, y=y.numpy(),
                        y_stream=ys.numpy(), h0_buf2=st["gridnet_bufs"]["buf2"]["h0"].numpy(),
                        istft_buf=st["istft_buf"].numpy(), wsum=weight_checksum(net.state_dict()))
    # ---- separation: longer than the attention window (T = 70 > 50), B=1, keep only a digest ---
    N2 = 128 * 70
    x2, _ = synth.mixture(1, N2, seed0=1100)
    e2 = synth.embedding(1, seed0=3100)
    with torch.no_grad():
        y2 = net(x2, e2)
    np.savez_compressed(os.path.join(HERE, "sep_golden_long.npz"), seed=seed, N=N2, y_tail=y2[..., -1024:].numpy(),
                        y_rms=float(y2.pow(2).mean().sqrt()), y_sum=float(y2.double().sum()))
    # ---- enrollment ------------------------------------------------------------------------------
    en = rl.reference_embed_net(seed)
    xe = synth.enrollment(2, 4800)
    with torch.no_grad():
        emb = en(xe)
    np.savez_compressed(os.path.join(HERE, "embed_golden.npz"), seed=seed, n=4800, emb=emb.numpy(),
                        wsum=weight_checksum(en.state_dict()))
    # ---- state_dict key names and shapes of both reference modules (checkpoint compatibility, SURVEY 8f-1) ----
    import json
    keys = {"sep": {k: list(v.shape) for k, v in net.state_dict().items()},
            "embed": {k: list(v.shape) for k, v in en.state_dict().items()}}
    with open(os.path.join(HERE, "ckpt_keys.json"), "w") as f:
        json.dump(keys, f, indent=0, sort_keys=True)
    reference_pins()
    print("written", os.listdir(HERE))


def reference_pins():
    """ref_pins.npz: what tests/test_oracle.py and tests/test_ckpt.py compare with the reference, recorded from it.
    Tensors too large to store whole are pinned by a sample and their norm (oracle/golden.py)."""
    import importlib
    p = {}
    # seeded default init of both networks (test_seeded_init_matches_reference, the checkpoint tests)
    for seed in (0, 11, 13):
        p.update(golden.fingerprint(f"init_sep_{seed}", rl.reference_net(seed).state_dict()))
    p.update(golden.fingerprint("init_embed_12", rl.reference_embed_net(12).state_dict()))
    # parameters: names and sizes (test_param_counts)
    for name, mod in (("sep", rl.reference_net(0)), ("embed", rl.reference_embed_net(0))):
        params = list(mod.named_parameters())
        p[f"params_{name}.names"] = np.array([k for k, _ in params])
        p[f"params_{name}.numel"] = np.array([v.numel() for _, v in params], dtype=np.int64)
    # whole-utterance output and the final streaming state (test_restatement_equals_reference_forward_and_state)
    net = rl.reference_net(3)
    x, _ = synth.mixture(2, 128 * 9 + 77, seed0=50)
    e = synth.embedding(2, seed0=60)
    with torch.no_grad():
        y = net(x, e)
        st = net.init_buffers(2, "cpu")
        _, st = net.predict(x, e[:, 0], st)
    p["fwd_state.wsum"] = weight_checksum(net.state_dict())
    p["fwd_state.y"] = y.numpy()
    for k in ("conv_buf", "deconv_buf", "istft_buf"):
        p.update(golden.pin(f"fwd_state.{k}", st[k]))
    for i in range(3):
        for k in ("K_buf", "V_buf", "h0", "c0"):
            p.update(golden.pin(f"fwd_state.buf{i}.{k}", st["gridnet_bufs"][f"buf{i}"][k]))
    # fp32 reference output the fp64 restatement is held to (test_restatement_fp64_floor)
    net = rl.reference_net(1)
    x, _ = synth.mixture(1, 128 * 8)
    e = synth.embedding(1)
    with torch.no_grad():
        p["fp64_floor.y"] = net(x, e).numpy()
    p["fp64_floor.wsum"] = weight_checksum(net.state_dict())
    # enrollment network (test_embed_restatement_equals_reference)
    en = rl.reference_embed_net(2)
    with torch.no_grad():
        p["embed.emb"] = en(synth.enrollment(2, 5000)).numpy()
    p["embed.wsum"] = weight_checksum(en.state_dict())
    # the STFT the reference vendors (test_stft_shim_equals_the_stft_the_reference_vendors)
    stft = importlib.import_module("src.models.tfgridnet_orig.stft").Stft
    for j, (n_fft, hop, n) in enumerate(((128, 64, 5000), (128, 64, 4999), (192, 128, 3001))):
        x = synth.enrollment(3, n).transpose(1, 2).contiguous()
        out, olens = stft(n_fft=n_fft, win_length=n_fft, hop_length=hop, window="hann")(x, torch.tensor([n, n, n]))
        p.update(golden.pin(f"stft{j}", out, n=1024))
        p[f"stft{j}.olens"] = olens.numpy()
    # separator output behind a checkpoint written from the reference (test_checkpoint_outputs_on_gpu)
    net = rl.reference_net(13)
    x, _ = synth.mixture(1, 128 * 12)
    with torch.no_grad():
        p["ckpt_gpu.y"] = net(x, synth.embedding(1)).numpy()
    np.savez_compressed(os.path.join(HERE, "ref_pins.npz"), **p)


if __name__ == "__main__":
    main()
