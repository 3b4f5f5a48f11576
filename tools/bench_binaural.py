"""Time l2h_eval_binaural (ILD + ITD in one pass) with CUDA events and report it against the B200's copy peak and its
FP32 FMA rate.  python tools/bench_binaural.py [--iters 200] [--out profiles/r03a_binaural_bench.json]

Shapes: B = 256 x 64 000 (4 s at 16 kHz, static and moving) and the evaluation batch B = 4 x 80 000.  At B = 256 the
inputs (est + gt, 262 MB) exceed the 126 MB L2, so every timed call reads them from HBM; at B = 4 (5 MB) they stay in L2.
Algorithmic bytes = 16 B T (two fp32 signals of two ears); FMAs = 2 B T (2 t + 1) (est and gt, every lag).
The copy peak is the measured HBM copy rate the project's rooflines use (DESIGN.md section 4.3); the FMA peak is
127 FMA/clk/SM (tools/ffma_microbench.cu) x 148 SMs x the card's maximum SM clock, read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from lookoncetohear_b200.metrics import binaural_errors, frame_width, max_lag  # noqa: E402

COPY_PEAK_GBS = 6590.9
FMA_PER_CLK_SM = 127


def card():
    info = {"name": torch.cuda.get_device_name(0), "sms": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"] = float(q[0])
        info["max_sm_clock_mhz"] = float(q[1])
    except Exception as exc:                                   # the numbers stay, the clock-based bound is then omitted
        info["query_error"] = repr(exc)
    return info


def run(B, T, sr, moving, iters, info):
    gen = torch.Generator(device="cuda").manual_seed(B + T)
    est = 0.1 * torch.randn(B, 2, T, generator=gen, device="cuda")
    gt = 0.1 * torch.randn(B, 2, T, generator=gen, device="cuda")
    for _ in range(10):
        binaural_errors(est, gt, sr, moving)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        binaural_errors(est, gt, sr, moving)
    t1.record()
    torch.cuda.synchronize()
    us = t0.elapsed_time(t1) * 1e3 / iters
    L = frame_width(sr) if moving else T
    t = min(max_lag(sr), L // 2)
    nbytes = 16 * B * T
    fmas = 2 * B * T * (2 * t + 1)
    row = {"B": B, "T": T, "sr": sr, "mode": "moving" if moving else "static", "iters": iters, "us_per_call": round(us, 2),
           "bytes": nbytes, "GB_per_s": round(nbytes / us / 1e3, 1), "frac_copy_peak": round(nbytes / us / 1e3 / COPY_PEAK_GBS, 3),
           "fma": fmas, "TFMA_per_s": round(fmas / us / 1e6, 2)}
    t_bytes = nbytes / (COPY_PEAK_GBS * 1e3)                    # us at the copy peak
    if "max_sm_clock_mhz" in info:
        peak = FMA_PER_CLK_SM * info["sms"] * info["max_sm_clock_mhz"] * 1e6
        row["frac_fma_peak"] = round(fmas / (us * 1e-6) / peak, 3)
        t_fma = fmas / peak * 1e6
        row["bound"] = "fma" if t_fma > t_bytes else "hbm"
        row["frac_of_bound"] = round(max(t_fma, t_bytes) / us, 3)
    # wall time includes the wrapper (workspace allocation from the cache, two launches)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03a_binaural_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_binaural needs a GPU")
    info = card()
    rows = [run(256, 64000, 16000, False, a.iters, info), run(256, 64000, 16000, True, a.iters, info),
            run(4, 80000, 16000, False, a.iters, info), run(4, 80000, 16000, True, a.iters, info)]
    res = {"card": info, "copy_peak_GBs": COPY_PEAK_GBS, "rows": rows}
    for r in rows:
        print(json.dumps(r))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("card", json.dumps(info))


if __name__ == "__main__":
    main()
