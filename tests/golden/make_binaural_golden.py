"""Generate tests/golden/binaural_golden.npz from the REFERENCE ITSELF (run where a checkout of the reference exists, see
oracle/ref_loader.py):  python tests/golden/make_binaural_golden.py

Its own script, so that regenerating it never rewrites the other fixtures.  The inputs are not stored: they are
regenerated from seeds by tests/binaural_oracle.py::cases(), and a checksum of them is stored so that a drift of the
generator is detected rather than misread as a parity failure.  For every case and both modes (static, moving) the
file holds what src/eval/binaural.py returns -- ild_diff, itd_diff per mixture -- and, per window, chunk_and_mask's
validity, compute_ild's ILD, compute_itd's lag, and the two lags with the largest |correlation| of axiswise_xcorr with
their margin relative to ||left|| ||right|| (to tell near-ties, where float32 FFT rounding may pick either, from real
answers).
"""
import importlib.util
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
import binaural_oracle as bo  # noqa: E402
from oracle import ref_loader as rl  # noqa: E402


def reference_binaural():
    root = rl.reference_root()
    if root is None:
        raise RuntimeError("reference checkout not present")
    spec = importlib.util.spec_from_file_location("ref_binaural", os.path.join(root, "src", "eval", "binaural.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def binaural_pins():
    ref = reference_binaural()
    p = {}
    for name, (sr, e, g) in bo.cases().items():
        p[f"{name}.sr"] = np.int64(sr)
        p[f"{name}.est_sum"], p[f"{name}.gt_sum"] = bo.checksum(e), bo.checksum(g)
        _, TMAX = bo.frame_tmax(sr)
        for moving in (False, True):
            k = f"{name}.{'moving' if moving else 'static'}"
            p[k + ".ild_diff"] = np.asarray(ref.ild_diff(e, g, sr, moving=moving), dtype=np.float64)
            p[k + ".itd_diff"] = np.asarray(ref.itd_diff(e, g, sr, moving=moving), dtype=np.float64)
            if moving:
                ec, gc, mask = ref.chunk_and_mask(e, g, sr)              # [C, B, 2, FW], [C, B]
                ec, gc, mask = ec.transpose(1, 0, 2, 3), gc.transpose(1, 0, 2, 3), mask.T
            else:
                ec, gc, mask = e[:, None], g[:, None], np.ones((e.shape[0], 1), dtype=bool)
            p[k + ".valid"] = mask
            for tag, x in (("est", ec), ("gt", gc)):
                left, right = x[..., 0, :], x[..., 1, :]
                p[k + f".ild_{tag}"] = np.asarray(ref.compute_ild(left, right), dtype=np.float64)
                tau = np.rint(ref.compute_itd(left, right, sr, TMAX) * sr / 1e6).astype(np.int64)
                corr = ref.axiswise_xcorr(left, right)
                n = corr.shape[-1]
                t = min(TMAX, n // 2)
                a = np.abs(corr[..., np.arange(-t, t + 1) % n]).astype(np.float64)
                top1 = a.argmax(-1)
                assert np.array_equal(top1 - t, tau), (name, tag)
                best = np.take_along_axis(a, top1[..., None], -1)[..., 0]
                np.put_along_axis(a, top1[..., None], -1.0, -1)
                top2 = a.argmax(-1)
                second = np.take_along_axis(a, top2[..., None], -1)[..., 0]
                nrm = np.sqrt((left.astype(np.float64) ** 2).sum(-1) * (right.astype(np.float64) ** 2).sum(-1))
                with np.errstate(divide="ignore", invalid="ignore"):
                    p[k + f".margin_{tag}"] = np.where(nrm > 0, (best - second) / nrm, 0.0)
                p[k + f".tau_{tag}"] = tau
                p[k + f".top2_{tag}"] = np.stack([top1 - t, top2 - t], -1)
    p["cases"] = np.array(sorted(bo.cases()))
    np.savez_compressed(os.path.join(HERE, "binaural_golden.npz"), **p)


if __name__ == "__main__":
    binaural_pins()
    print("written", os.path.join(HERE, "binaural_golden.npz"))
