"""The reference's evaluation loop (src/ts_hear_test.py:93-166) with every arithmetic step on the GPU engine:

    mono events + impulse responses --render_binaural--> mixture, target          (multi_ch_simulator.py:56-58,
                                                                                     MixLibriSpeechNoisyEnrollNorm.py:179-202)
    enrollment recording --EmbedTFGridNet--> embedding                             (ts_hear_test.py:133-135)
    model(mixture, embedding) --Net--> outputs                                     (ts_hear_test.py:138)
    eval_metrics(outputs, target, mixture, embedding, embedding_gt)                (ts_hear_test.py:139-146)
    binaural_errors(outputs, target, sr, moving)  ILD / ITD errors                  (src/eval/binaural.py:49-149)

Synthetic inputs (no dataset in the image): white-noise events, exponentially decaying random impulse responses.  Only the
metric floats per mixture leave the device.  Usage: python examples/eval_gpu.py [n_batches] [batch]"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from lookoncetohear_b200 import EmbedTFGridNet, Net
from lookoncetohear_b200.configs import EMBED_PARAMS, TSH_PARAMS
from lookoncetohear_b200.metrics import binaural_errors, eval_metrics
from lookoncetohear_b200.render import render_binaural


def synthetic_batch(batch, n_src, n, rir_len, gen, dev):
    srcs = 0.1 * torch.randn(batch, n_src, n, generator=gen, device=dev)
    decay = torch.exp(-torch.arange(rir_len, device=dev) / (rir_len / 6.0))
    rirs = torch.randn(batch, n_src, 2, rir_len, generator=gen, device=dev) * decay
    noise = 0.02 * torch.randn(batch, 2, n, generator=gen, device=dev)
    scale = 0.5 + torch.rand(batch, generator=gen, device=dev)
    return srcs, rirs, noise, scale


def main():
    n_batches = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    batch = int(sys.argv[2]) if len(sys.argv) > 2 else 4            # ts_hear_test.py uses a DataLoader with batch_size 4
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    model = Net(**TSH_PARAMS).eval().to(dev)
    enroll_model = EmbedTFGridNet(**EMBED_PARAMS).eval().to(dev)
    gen = torch.Generator(device=dev).manual_seed(1)
    rows = []
    t0 = time.perf_counter()
    with torch.no_grad():
        for _ in range(n_batches):
            srcs, rirs, noise, scale = synthetic_batch(batch, 3, 80000, 200, gen, dev)
            events, mixture, _ = render_binaural(srcs, rirs, noise, scale)
            target = events[:, 0]                                              # tgt_idx = 0
            # noisy enrollment: the target speaker's other utterance rendered with another response, plus background
            e_src, e_rir, e_noise, e_scale = synthetic_batch(batch, 1, 80000, 200, gen, dev)
            _, enrollment, _ = render_binaural(e_src, e_rir, e_noise, e_scale)
            embedding = enroll_model(enrollment).unsqueeze(1)                  # [B, 1, 256]
            embedding_gt = torch.nn.functional.normalize(torch.rand(batch, 1, 256, generator=gen, device=dev), dim=-1)
            outputs = model(mixture, embedding)
            rows.append(torch.cat([eval_metrics(outputs, target, mixture, embedding, embedding_gt),
                                   binaural_errors(outputs, target, 16000),                 # static, whole 5 s
                                   binaural_errors(outputs, target, 16000, moving=True)], 1))   # 250 ms windows
    res = torch.cat(rows).cpu()                                                # the only device -> host copy
    dt = time.perf_counter() - t0
    print("output_sisnr  si_snr_i  embedding_sim  ild_diff_dB  itd_diff_us  ild_diff_moving  itd_diff_moving")
    print(res)
    print(f"{res.shape[0]} mixtures of 5 s in {dt:.2f} s wall (first call includes weight upload); Average SI-SNRi {res[:, 1].mean():.3f}")


if __name__ == "__main__":
    main()
