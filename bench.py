#!/usr/bin/env python
"""bench.py -- the reference's headline metric on B200: separated frames/s (8 ms hops of a 16 kHz
binaural stream) and the real-time factor, for BASELINE.json configs[1]: separation in 8 ms chunks,
batch 1, fp32, one stream per GPU.

A *step* = one pass of the hot path over one synthetic 4 s binaural mixture (500 hops) per GPU with a
fresh state (state init is inside the step).  Every hop is its own one-hop kernel chain with the
streaming state carried hop to hop, but -- read this -- `value` is BUFFERED-CLIP THROUGHPUT: the whole
clip is resident when the step starts and the 500 one-hop chains run as one wavefront-pipelined CUDA
graph (hop t+1 starts before hop t has finished), which needs the future audio to be there already.
The strictly causal figures (hop t+1 not started before hop t is out) are reported on the same line
under `streaming_causal`: frames/s, real-time factor, single-chunk latency, and an end-to-end variant
that copies every 8 ms chunk host->device and its output back per hop.
`value` = hops/s over all ranks with the clip resident in HBM (l2h_sep_stream_dev); `e2e` = the same
through the C-ABI host-buffer call (l2h_sep_stream_host): per round of up to 500 hops ONE host->device
copy of the round's samples from pinned memory and ONE device->host copy of its output, inside the
timed region.  Further blocks on the line: `batched_streaming` (configs[4] per-GPU shape, 256 streams
per rank, at every N), `offline_bf16_256` (configs[2]), `enrollment_1024` (configs[3]).
`--impl reference` times the reference's own CPU path (the reference modules when the checkout is
present, else the oracle port) on the host cores with the same workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--chunks-per-call C] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

`--dump-outputs DIR` writes what the last timed step of each arm handed back to its caller (rank 0), float32:
y.npy (the separated clip of the device-resident arm), state.*.npy (its streaming state after the clip, in the
reference's layout, SepState.to_reference) and y_e2e.npy (the clip of the host-buffer arm).  Inputs and weights
are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

CLIP_SAMPLES = 64000          # 4 s @ 16 kHz (configs[0]/[1]: "single 4 s binaural mixture")
HOP = 128
FRAMES = CLIP_SAMPLES // HOP  # 500
METRIC = ("separated frames/sec (8 ms chunks, 16 kHz binaural, batch 1 per GPU): buffered-clip throughput, the one-hop chains "
          "of a resident clip pipelined as a wavefront; strictly causal figures under streaming_causal")
# SURVEY.md 8(d): algorithmic work per hop per stream
FLOP_PER_FRAME = 74.67e6
BYTES_PER_FRAME = 5.50e6


def workload_name():
    return ("streaming separation, 8 ms chunks, batch=1 per GPU, fp32 (BASELINE configs[1]); %.1f s clip = %d hops per step, "
            "fresh state per step" % (FRAMES * 0.008, FRAMES))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d.get("bf16_tflops_sustained", 1412.4), source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                 0x80: "hw_power_brake_slowdown"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def time_cpu_streaming(frames, chunks_per_call, passes, threads, seed=0):
    """The CPU path on the host cores: chunked predict(pad=False) over `frames` hops, B=1.
    Uses the reference's own modules when the checkout exists, else the oracle port."""
    from lookoncetohear_b200 import Net, synth
    from lookoncetohear_b200.configs import TSH_PARAMS
    from oracle import ref_loader, restate
    torch.set_num_threads(threads)
    x, _ = synth.mixture(1, frames * HOP)
    e = synth.embedding(1)[:, 0]
    xp = torch.nn.functional.pad(x, (0, 64))
    step = HOP * chunks_per_call
    if ref_loader.available():
        kind = "reference"
        net = ref_loader.reference_net(seed)

        def one_pass():
            st = net.init_buffers(1, "cpu")
            for i in range(0, frames, chunks_per_call):
                net.predict(xp[..., HOP * i:HOP * i + step + 64], e, st, pad=False)
    else:
        kind = "port"
        restate.set_fast(True)            # ATen's fused LSTM, like the reference's nn.LSTM
        torch.manual_seed(seed)
        sd = {k: v.detach().clone() for k, v in Net(**TSH_PARAMS).state_dict().items()}

        def one_pass():
            st = restate.sep_init_state(sd, 1)
            for i in range(0, frames, chunks_per_call):
                restate.sep_predict(sd, xp[..., HOP * i:HOP * i + step + 64], e, st, pad=False)
    best = None
    with torch.no_grad():
        for _ in range(passes):
            t0 = time.perf_counter()
            one_pass()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return frames / best, kind, best



# SURVEY.md 8(d): FLOPs per hop per stream that run as tensor-core GEMMs in the batched / offline paths
# (per block: W_ih of both LSTMs 6.36 + 3.18, the two Linears 1.59 + 0.79, Q|K|V 1.39 MFLOP) x 3 blocks
TC_FLOP_PER_FRAME = 3 * (6.36 + 3.18 + 1.59 + 0.79 + 1.39) * 1e6
EMBED_FLOP_PER_UTT = 255e9            # 5 s utterance, SURVEY.md section 2.1
EMBED_TC_FLOP_PER_UTT = 255e9 - 31e9  # everything except the recurrent h W_hh products (CUDA cores)


def _dev_time(fn, reps, sync):
    """best-of-`reps` device time (ms) of fn() with CUDA events"""
    best = None
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        sync()
        ms = a.elapsed_time(b)
        best = ms if best is None else min(best, ms)
    return best


def measure_batched_streaming(net, dev, rank, nb=256, nsteps=60):
    """BASELINE configs[4] per-GPU shape: `nb` independent streams advancing one 8 ms hop per step (this rank's
    share of the 2048).  Returns (ms for nsteps-10 steps, state GB)."""
    from lookoncetohear_b200 import synth
    g = torch.Generator().manual_seed(5000 + rank)
    xb = (0.1 * torch.randn(nb, 2, HOP * nsteps, generator=g)).to(dev)
    eb = synth.embedding(8, seed0=6000 + rank)[:, 0].repeat(nb // 8, 1).to(dev)
    yb = torch.empty(nb, 2, HOP * nsteps, device=dev)
    best, stb = None, None
    for it in range(3):
        stb = net.init_buffers(nb, dev)
        net.stream_dev(xb, eb, chunks_per_call=1, state=stb, n_calls=10, out=yb)     # warm (gate build, graph)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        net.stream_dev(xb[..., HOP * 10:], eb, chunks_per_call=1, state=stb, n_calls=nsteps - 10, out=yb[..., HOP * 10:])
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        best = ms if best is None else min(best, ms)
    gb = stb.buf.numel() * stb.buf.element_size() / 1e9
    return best, gb


def measure_offline_bf16(net, dev, nb=256):
    """BASELINE configs[2]: nb clips of 4 s in one forward(), bf16 tensor-core operands."""
    g = torch.Generator().manual_seed(7000)
    x = (0.1 * torch.randn(nb, 2, CLIP_SAMPLES, generator=g)).to(dev)
    e = torch.rand(nb, 1, 256, generator=g).to(dev)
    e = e / e.norm(dim=-1, keepdim=True)
    net.set_option("bf16", 1)
    try:
        with torch.no_grad():
            net(x[:32], e[:32])
            torch.cuda.synchronize()
            ms = _dev_time(lambda: net(x, e), 2, torch.cuda.synchronize)
    finally:
        net.set_option("bf16", 0)
    return ms


def measure_enrollment(dev, nb=1024, n=80000):
    """BASELINE configs[3]: nb five-second utterances through EmbedTFGridNet.forward (device-resident input)."""
    from lookoncetohear_b200 import EmbedTFGridNet
    from lookoncetohear_b200.configs import EMBED_PARAMS
    torch.manual_seed(0)
    net = EmbedTFGridNet(**EMBED_PARAMS).eval().to(dev)
    g = torch.Generator().manual_seed(8000)
    x = (0.1 * torch.randn(64, 2, n, generator=g)).repeat(nb // 64, 1, 1)
    x = (x * torch.linspace(0.5, 2.0, nb)[:, None, None]).to(dev)
    with torch.no_grad():
        net(x[:64])
        torch.cuda.synchronize()
        ms = _dev_time(lambda: net(x), 2, torch.cuda.synchronize)
    del net
    return ms


DUMP_BYTES = 60e6       # --dump-outputs thins above this; the per-row rounding of the thinning keeps it under 64 MB


def step_outputs(net, y, st):
    """Host copies of what a device-resident step hands its caller: the separated clip `y` and the streaming state `st`,
    the state converted to the reference's layout on a host copy (no device memory is allocated)."""
    from lookoncetohear_b200.net import SepState
    ref = SepState(st.buf.cpu(), st.batch, st.n_blocks, *net._state_layout()).to_reference()
    out = {"y": y.cpu()}
    out.update({f"state.{k}": ref[k] for k in ("conv_buf", "deconv_buf", "istft_buf")})
    for b, bufs in ref["gridnet_bufs"].items():
        out.update({f"state.{b}.{k}": v for k, v in bufs.items()})
    return out


def write_outputs(out_dir, arrays):
    """out_dir/<name>.npy in float32 for every array.  Should they come to more than DUMP_BYTES (a long --clip-hops),
    every array keeps every k-th element of its last axis, the same k for all."""
    import math

    import numpy as np
    k = max(1, math.ceil(sum(4 * t.numel() for t in arrays.values()) / DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t[..., ::k].float().numpy())


def run_reference(args, rank, world):
    if rank != 0:
        return
    # each step = a bounded sample of the workload: 125 hops (1 s of audio) of the same clip, chunked.
    # Chunk-by-chunk streaming on CPU is dispatch-bound and often fastest on ONE thread (SURVEY.md
    # section 6), so probe 1 thread vs all cores first and run the timed steps on the faster setting.
    sample_frames = 125
    allc = os.cpu_count() or 1
    probe = {t: time_cpu_streaming(4, args.chunks_per_call, 1, t)[0] for t in sorted({1, min(allc, 8)})}
    threads = max(probe, key=probe.get)
    times = []
    kind = None
    for i in range(args.warmup + args.steps):
        fps, kind, dt = time_cpu_streaming(sample_frames, args.chunks_per_call, 1, threads)
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = sample_frames * len(times) / total
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rtf": value / 125.0,
        "config": {"workload": workload_name(), "chunks_per_call": args.chunks_per_call,
                   "sample": f"bounded sample: {sample_frames} hops (1 s) of the same 4 s clip per step, strictly hop by hop on the CPU"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": kind,
                         "sample": f"{sample_frames} hops of the 4 s clip per step, chunked predict(pad=False), "
                                   f"{cpu_model_name()}"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunks-per-call", type=int, default=1,
                    help="hops handed to the engine per call (1 = true chunk-by-chunk streaming)")
    ap.add_argument("--no-extras", action="store_true", help="skip the latency / buffered-throughput extras")
    ap.add_argument("--clip-hops", type=int, default=0,
                    help="profiling aid: shorten the clip to this many hops (the default, 0, is the 4 s = 500-hop clip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32), see the module docstring")
    args = ap.parse_args()

    global CLIP_SAMPLES, FRAMES
    if args.clip_hops > 0:
        FRAMES = args.clip_hops
        CLIP_SAMPLES = FRAMES * HOP
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from lookoncetohear_b200 import Net, _cabi, build, synth
    from lookoncetohear_b200.configs import TSH_PARAMS

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    build.build()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"       # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)

    # ---- weights: rank 0 owns them, NCCL broadcast to the other ranks ---------------------------
    torch.manual_seed(0 if rank == 0 else 12345 + rank)      # non-zero ranks start with different values
    net = Net(**TSH_PARAMS).eval().to(dev)
    emb = synth.embedding(1, seed0=3000)[:, 0].to(dev)
    if world > 1:
        for t in list(net.parameters()) + list(net.buffers()):
            dist.broadcast(t.data, src=0)
        dist.broadcast(emb, src=0)
        net.refresh_weights()

    cpc = args.chunks_per_call
    n_calls = (FRAMES + cpc - 1) // cpc
    x_cpu, _ = synth.mixture(1, CLIP_SAMPLES, seed0=1000 + rank)
    x_dev = x_cpu.to(dev)
    x_pin = x_cpu.pin_memory()
    y_dev = torch.empty(1, 2, CLIP_SAMPLES, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)      # 256 MiB > 126 MB L2
    L = _cabi.lib()

    def step_dev():
        st = net.init_buffers(1, dev)
        net.stream_dev(x_dev, emb, chunks_per_call=cpc, state=st, n_calls=n_calls, out=y_dev)

    y_pin = torch.empty(1, 2, n_calls * HOP * cpc, dtype=torch.float32).pin_memory()

    def step_host():
        return net.stream_host(x_pin, emb, chunks_per_call=cpc, out=y_pin)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm -------------------------------------------------------------------------
    for _ in range(args.warmup):
        step_dev()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    evs = []
    _cabi.check(L.l2h_sep_launch_count(net._engine(), None, 1))   # the engine counts its kernels (graph replays by node)
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.fill_(1.0)                                         # L2 flush between timed iterations
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step_dev()
        b.record()
        evs.append((a, b))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    n_launched = ctypes.c_int64()
    _cabi.check(L.l2h_sep_launch_count(net._engine(), ctypes.byref(n_launched), 0))
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    dump = None
    if args.dump_outputs and rank == 0:
        dump = step_outputs(net, y_dev, net._last_stream_state)    # stream_dev keeps the state of its last call
    # ---- end-to-end arm (host buffers, H2D/D2H inside) -----------------------------------------------
    for _ in range(min(args.warmup, 2)):
        step_host()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        y_host = step_host()
    e1.record()
    barrier()
    e2e_wall = time.perf_counter() - t0
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * e2e_wall)          # the call ends with a stream sync; take the larger
    clocks = sampler.result()
    if dump is not None:
        dump["y_e2e"] = y_host
        write_outputs(args.dump_outputs, dump)

    # ---- configs[4] per-GPU shape on EVERY rank: 256 streams per rank, one hop per step, max-over-ranks time ----
    bs_ms, bs_gb, bs_err = 0.0, 0.0, None
    NB_STREAMS, NB_STEPS = 256, 60
    if not args.no_extras:
        try:
            bs_ms, bs_gb = measure_batched_streaming(net, dev, rank, NB_STREAMS, NB_STEPS)
        except Exception as exc:                                   # never let a block break the bench line
            bs_err = repr(exc)[:200]
            bs_ms = float("inf")
    barrier()
    tm = torch.tensor([dev_ms, e2e_ms, bs_ms], device=dev, dtype=torch.float64)
    nl = torch.tensor([n_launched.value], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(nl, op=dist.ReduceOp.SUM)             # kernels of the whole job
    dev_ms, e2e_ms, bs_ms = float(tm[0]), float(tm[1]), float(tm[2])
    frames_total = world * FRAMES * args.steps
    value = frames_total / (dev_ms * 1e-3)
    e2e_value = frames_total / (e2e_ms * 1e-3)

    # host<->device bytes of one step through l2h_sep_stream_host (rounds of `hops_per_round` hops)
    hops_per_round = max(cpc, net.pipeline_frames() if cpc == 1 else 1)
    h2d_bytes = d2h_bytes = 0
    for h0 in range(0, n_calls * cpc, hops_per_round):
        hops = min(hops_per_round, n_calls * cpc - h0)
        h2d_bytes += 2 * max(0, min(CLIP_SAMPLES - h0 * HOP, HOP * hops + 64)) * 4
        d2h_bytes += 2 * max(0, min(CLIP_SAMPLES - h0 * HOP, HOP * hops)) * 4
    extras = {}
    roof = None
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_extras:          # extras are single-GPU figures (the N > 1 line carries value / e2e / roofline)
        # single-chunk latency: one call, synchronised, median of 200 (graph replay)
        st = net.init_buffers(1, dev)
        lat = []
        net.stream_dev(x_dev, emb, chunks_per_call=1, state=st, n_calls=60, out=y_dev)
        torch.cuda.synchronize()
        lat_dev = []
        for i in range(200):
            ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            ea.record()
            net.stream_dev(x_dev[..., :HOP * 8], emb, chunks_per_call=1, state=st, n_calls=1, out=y_dev[..., :HOP * 8])
            eb.record()
            torch.cuda.synchronize()
            lat.append(time.perf_counter() - t0)
            lat_dev.append(ea.elapsed_time(eb))
        extras["chunk_latency_us"] = 1e6 * statistics.median(lat)          # host wall clock: call + graph launch + sync
        extras["chunk_latency_device_us"] = 1e3 * statistics.median(lat_dev)   # CUDA events around the same call
        # the same 500-hop stream with the hops run strictly one after the other (no wavefront pipelining)
        net.set_option("pipeline", 0)
        for it in range(3):
            st = net.init_buffers(1, dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            net.stream_dev(x_dev, emb, chunks_per_call=1, state=st, n_calls=FRAMES, out=y_dev)
            b.record()
            torch.cuda.synchronize()
            extras["frames_per_s_unpipelined"] = FRAMES / (a.elapsed_time(b) * 1e-3)
        net.set_option("pipeline", 1)
        # buffered throughput: more hops per call (latency traded for throughput), same clip, same state API
        buf = {}
        for c in (4, 20, 500):
            nc = (FRAMES + c - 1) // c
            for it in range(3):
                st = net.init_buffers(1, dev)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                net.stream_dev(x_dev, emb, chunks_per_call=c, state=st, n_calls=nc, out=y_dev)
                b.record()
                torch.cuda.synchronize()
                buf[str(c)] = FRAMES / (a.elapsed_time(b) * 1e-3)
        extras["frames_per_s_by_chunks_per_call"] = buf
        # strictly causal streaming END TO END: per hop one H2D of the 8 ms chunk (+ look-ahead) from pinned memory,
        # one predict() call, one D2H of the 128 output samples per ear -- what a live caller does
        try:
            hops = 150
            xin = torch.nn.functional.pad(x_cpu[..., :HOP * hops], (0, 64)).pin_memory()
            yout = torch.empty(1, 2, HOP * hops).pin_memory()
            chunk = torch.empty(1, 2, HOP + 64).pin_memory()
            yhop = torch.empty(1, 2, HOP).pin_memory()
            st = net.init_buffers(1, dev)
            with torch.no_grad():
                for i in range(hops):
                    if i == 30:
                        torch.cuda.synchronize()
                        t0 = time.perf_counter()
                    chunk.copy_(xin[..., HOP * i:HOP * i + HOP + 64])       # the caller's pinned chunk buffer (host memcpy of 1.5 KB)
                    net.predict_host(chunk, emb, st, out=yhop)            # H2D + one-hop chain + D2H + stream sync, one C call
                    yout[..., HOP * i:HOP * (i + 1)].copy_(yhop)
            dt = time.perf_counter() - t0
            extras["e2e_causal_frames_per_s"] = (hops - 30) / dt
        except Exception as exc:
            extras["e2e_causal_frames_per_s"] = {"error": repr(exc)[:200]}
        extras["streaming_causal"] = {
            "frames_per_s": extras.get("frames_per_s_unpipelined"), "rtf": (extras.get("frames_per_s_unpipelined") or 0) / 125.0,
            "chunk_latency_device_us": extras.get("chunk_latency_device_us"), "chunk_latency_host_us": extras.get("chunk_latency_us"),
            "e2e_frames_per_s": extras.get("e2e_causal_frames_per_s"),
            "e2e_api": "per hop Net.predict_host (l2h_sep_stream_host with one call): pinned H2D of 192 samples x 2 mics, the one-hop chain, D2H of 128 samples x 2 ears, stream sync",
            "note": "hop t+1 is not started before hop t has finished: what a live 8 ms stream gets"}
        pkb = peaks()
        # ---- BASELINE configs[2]: offline batch of 256 x 4 s clips, bf16 tensor-core operands ----
        try:
            ms = measure_offline_bf16(net, dev, 256)
            fps = 256 * FRAMES / (ms * 1e-3)
            extras["offline_bf16_256"] = {
                "clips": 256, "clip_s": FRAMES * 0.008, "ms": ms, "frames_per_s": fps, "rtf_aggregate": fps / 125.0,
                "dtype": "bf16 weights on the tensor cores, activations as bf16 hi+lo (2 MMA passes), fp32 accumulate; fp32 recurrent "
                         "state / LayerNorm / element-wise",
                "tensor_tflops_algorithmic": fps * TC_FLOP_PER_FRAME / 1e12,
                "tensor_frac": fps * TC_FLOP_PER_FRAME / 1e12 / pkb["bf16_tflops"], "tflops_total_algorithmic": fps * FLOP_PER_FRAME / 1e12,
                "peak": pkb["bf16_tflops"], "peak_source": pkb["source"] + " bf16_tflops_sustained",
                "note": "53 % of the FLOPs are tensor-core GEMMs (W_ih, Linears, Q|K|V); the recurrences (h W_hh), the 50-frame "
                        "attention and the LayerNorms run on the CUDA cores"}
        except Exception as exc:
            extras["offline_bf16_256"] = {"error": repr(exc)[:200]}
        # ---- BASELINE configs[3]: enrollment, 1024 utterances of 5 s ----
        try:
            ms = measure_enrollment(dev, 1024)
            ups = 1024 / (ms * 1e-3)
            extras["enrollment_1024"] = {
                "utterances": 1024, "utt_s": 5.0, "ms": ms, "utt_per_s": ups, "tflops_algorithmic": ups * EMBED_FLOP_PER_UTT / 1e12,
                "dtype": "fp32 in/out; tensor-core GEMMs as bf16x3 split products (3 MMA passes per product)",
                "tensor_tflops_algorithmic": ups * EMBED_TC_FLOP_PER_UTT / 1e12,
                "tensor_frac_algorithmic": ups * EMBED_TC_FLOP_PER_UTT / 1e12 / pkb["bf16_tflops"],
                "tensor_frac_issued": 3 * ups * EMBED_TC_FLOP_PER_UTT / 1e12 / pkb["bf16_tflops"],
                "peak": pkb["bf16_tflops"], "peak_source": pkb["source"] + " bf16_tflops_sustained"}
        except Exception as exc:
            extras["enrollment_1024"] = {"error": repr(exc)[:200]}
    if rank == 0 and not args.no_extras:
        pkb = peaks()
        if bs_err is not None or bs_ms == float("inf"):
            extras["batched_streaming"] = {"error": bs_err or "a rank failed"}
        else:
            fps = world * NB_STREAMS * (NB_STEPS - 10) / (bs_ms * 1e-3)
            extras["batched_streaming"] = {
                "streams_per_gpu": NB_STREAMS, "streams_total": world * NB_STREAMS, "frames_per_s": fps, "rtf_aggregate": fps / 125.0,
                "ms_per_hop_step": bs_ms / (NB_STEPS - 10), "hbm_gbs_algorithmic_per_gpu": fps / world * BYTES_PER_FRAME / 1e9,
                "hbm_frac": fps / world * BYTES_PER_FRAME / 1e9 / pkb["hbm_gbs"], "peak_source": pkb["source"],
                "timing": "max over ranks of the device time of 50 hop-steps (best of 3), every rank its own 256 streams",
                "note": "state (%.2f GB per GPU) >> L2: every hop re-reads each stream's K/V rings from HBM; "
                        "algorithmic bytes 5.50 MB per hop per stream (SURVEY.md 8d)" % bs_gb}
    if rank == 0:
        # per-kernel device times of one streaming chain (CUDA events on the launching stream)
        prof = profile_chain(net, x_dev, emb, dev, cpc)
        pk = peaks()
        dom = max(prof.items(), key=lambda kv: kv[1]["ms_total"])
        # dominant kernel: algorithmic bytes per launch (DESIGN.md section 4) / its mean duration
        alg = kernel_algorithmic_bytes(dom[0], cpc)
        ach = alg / (dom[1]["ms_mean"] * 1e-3) / 1e9
        tr = trace_one_hop(net, x_dev, emb, dev)
        fps_seq = extras.get("frames_per_s_unpipelined")
        chain_us = 1e6 / fps_seq if fps_seq else tr["span_us"]      # device time per hop of back-to-back one-hop calls (chain + the gap between two graph launches)
        latency_model = {"serial_steps": 3 * 97, "t_step_floor_us": 0.23, "t_step_measured_us": tr["t_step_us"],
                         "chain_us": chain_us, "kernels_per_hop": tr["kernels"],
                         "latency_frac": 3 * 97 * 0.23 / chain_us, "recurrence_share_of_chain": 3 * 97 * (tr["t_step_us"] or 0.0) / chain_us,
                         "fma_pipe_pct_of_dominant_kernel": 15.6,
                         "source": "chain_us = 1e6 / frames_per_s_unpipelined (untraced); t_step, kernels and the timeline from the device-side "
                                   "trace of one one-hop call (l2h_sep_trace_*; with tracing on every kernel exit also flushes its time stamps)",
                         "traced_span_us": tr["span_us"], "timeline_us": tr["timeline_us"]}
        roof = {"bound": "hbm", "kernel": dom[0], "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": ach / pk["hbm_gbs"],
                # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel, from the committed
                # ncu --set full capture profiles/r01e_lstm_rec3_full.md (warm L2: the launch's 379 KB of
                # algorithmic bytes are L2 hits; 0.9 KB read + 10.5 KB written reach DRAM)
                "traffic": 11392.0 if dom[0] == "lstm_intra" else None, "peak_source": pk["source"],
                "alg_bytes_per_launch": alg, "mean_us_per_launch": 1e3 * dom[1]["ms_mean"],
                "share_of_chain": dom[1]["ms_total"] / sum(v["ms_total"] for v in prof.values()),
                # fma_pipe_pct from the ncu capture profiles/r01e_lstm_rec3_full.md
                # the model that governs batch 1: the chain cannot be shorter than its 3 x 97 dependent recurrent steps.
                # t_step_floor = 0.23 us: the FMA + shuffle + barrier floor of one 256x64 step on one SM
                # (profiles/r01c_lstm_microbench.txt); chain_us / t_step_measured from the device-side trace of one hop
                "latency_model": latency_model,
                "note": "batch-1 streaming is latency-bound (serial LSTM chain, 13 MB working set resident in L2); "
                        "whole-chain algorithmic rate: %.1f GB/s, %.2f TFLOP/s fp32" % (
                            value / world * BYTES_PER_FRAME / 1e9, value / world * FLOP_PER_FRAME / 1e12)}
        extras["kernel_us"] = {k: round(1e3 * v["ms_mean"], 2) for k, v in prof.items()}
        if world == 1 and not args.no_extras:
            allc = os.cpu_count() or 1
            # chunk-by-chunk streaming on CPU is dispatch-bound: more threads are slower (0.14 frames/s on 128
            # threads vs 190 on one, measured); probe 1 thread vs min(all, 8) briefly and keep the faster
            probe = {t: time_cpu_streaming(4, cpc, 1, t)[0] for t in sorted({1, min(allc, 8)})}
            threads = max(probe, key=probe.get)
            fps, kind, _ = time_cpu_streaming(125, cpc, 2, threads)
            cpu_base = {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind,
                        "sample": "125 hops (1 s) of the same clip, chunked predict(pad=False), best of 2, on the "
                                  f"faster of 1 thread / all cores; {cpu_model_name()}; host has {allc} cores",
                        "probe_frames_per_s_by_threads": {str(t): v for t, v in probe.items()}}
        out = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "rtf": value / world / 125.0,
            "config": {"workload": workload_name(),
                       "chunks_per_call": cpc,
                       "pipeline": "wavefront over (block, hop) stages: up to %d one-hop chains per multi-stream CUDA graph; every "
                                   "hop is its own T=1 kernel chain with the state carried hop to hop, results bit-identical to the "
                                   "sequential run (frames_per_s_unpipelined / chunk_latency_us give the strictly sequential "
                                   "figures)" % net.pipeline_frames(),
                       "parallelism": f"dp{world} (independent streams, weights broadcast over NCCL)",
                       "l2": "flushed (256 MiB write) between timed iterations"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "rtf": e2e_value / world / 125.0, "hops_per_round": hops_per_round,
                    "api": "l2h_sep_stream_host: pinned host clip in, pinned host clip out; per round one cudaMemcpy2DAsync "
                           "H2D of the round's samples, the one-hop kernel chains of the round, one D2H of its output -- all "
                           "inside the timed region, fresh state per step"},
            "gpu_launches": int(nl.item()),
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu_base, "wall_s": t_wall,
        }
        out.update(extras)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def kernel_algorithmic_bytes(name, cpc):
    """Algorithmic HBM bytes of one launch of a chain kernel at batch 1 (DESIGN.md section 4)."""
    rows = 97 * cpc
    if name == "lstm_intra":
        return rows * 512 * 4 + rows * 128 * 4 + 2 * 256 * 64 * 4
    if name == "lstm_inter":
        return rows * 256 * 4 + rows * 64 * 4 + 256 * 64 * 4 + 2 * 2 * 97 * 64 * 4
    if name == "attn":
        return cpc * 4 * (584 * 4 + 50 * (584 + 1552) * 4 + 1552 * 4) if cpc == 1 else \
            4 * ((49 + cpc) * (584 + 1552) * 4 + cpc * (584 + 1552) * 4)
    return rows * 64 * 4 * 2


TRACE_NAMES = ["front", "gemm_ih", "lstm", "mid_a", "mid_b", "mid_c", "qkv", "attn", "attn_out", "back", "mid", "tail"]


def trace_one_hop(net, x_dev, emb, dev, reps=7):
    """Device-side timeline of ONE one-hop chain (the latency path) from the engine's trace (l2h_sep_trace_start/_read:
    the first thread of every kernel stores %globaltimer at entry / exit, the BiLSTM also around its 97-step loop).
    Returns the median run: span of the chain, kernels in it, the recurrence's measured time per step."""
    import numpy as np
    from lookoncetohear_b200 import _cabi
    L = _cabi.lib()
    REC = np.dtype([("t0", "<u8"), ("t1", "<u8"), ("ptr", "<u8"), ("kernel", "<u4"), ("sm", "<u4")])
    st = net.init_buffers(1, dev)
    need = HOP * (56 + reps + 1)
    if x_dev.shape[-1] < need:                  # short clips (--clip-hops): tile the audio, the timeline does not depend on the samples
        x_dev = x_dev[:1].repeat(1, 1, (need + x_dev.shape[-1] - 1) // x_dev.shape[-1])
    x_dev = x_dev[:1].contiguous()
    emb = emb[:1].contiguous()
    y = torch.empty(1, 2, x_dev.shape[-1], device=dev)
    for h in range(56):                         # rings full, graph instantiated
        net.stream_dev(x_dev[..., HOP * h:], emb, chunks_per_call=1, state=st, n_calls=1, out=y[..., HOP * h:])
    runs = []
    for r in range(reps):
        h = 56 + r
        _cabi.check(L.l2h_sep_trace_start(net._engine(), 256))
        torch.cuda.synchronize()
        net.stream_dev(x_dev[..., HOP * h:], emb, chunks_per_call=1, state=st, n_calls=1, out=y[..., HOP * h:])
        torch.cuda.synchronize()
        buf = np.zeros(256, dtype=REC)
        n = ctypes.c_int32()
        _cabi.check(L.l2h_sep_trace_read(net._engine(), buf.ctypes.data_as(ctypes.c_void_p), 256, ctypes.byref(n)))
        rec = buf[:n.value]
        rec = rec[rec["t1"] > 0]
        ker = rec[rec["kernel"] < 100]
        ker = ker[np.argsort(ker["t0"])]
        org = int(ker["t0"].min())
        marks = rec[rec["kernel"] >= 100]
        loop0 = np.sort(marks["t0"][marks["kernel"] == 100 + 20 * 2 + 0])     # BiLSTM: loop start / end
        loop1 = np.sort(marks["t0"][marks["kernel"] == 100 + 20 * 2 + 1])
        steps = [(int(b) - int(a)) / 1e3 / 97.0 for a, b in zip(loop0, loop1)]
        runs.append({"span_us": (int(ker["t1"].max()) - org) / 1e3, "kernels": int(len(ker)),
                     "t_step_us": float(np.median(steps)) if steps else None,
                     "timeline_us": [[TRACE_NAMES[min(int(k["kernel"]), 11)], round((int(k["t0"]) - org) / 1e3, 1), round((int(k["t1"]) - org) / 1e3, 1)] for k in ker]})
    _cabi.check(L.l2h_sep_trace_start(net._engine(), 0))
    runs.sort(key=lambda d: d["span_us"])
    return runs[len(runs) // 2]


def profile_chain(net, x_dev, emb, dev, cpc, iters=20, batch=1):
    """Times every kernel of the chain with CUDA events (l2h_sep_profile) -> {name: {ms_mean, ms_total}}."""
    from lookoncetohear_b200 import _cabi
    L = _cabi.lib()
    net._sync_weights(dev)
    st = net.init_buffers(batch, dev)
    ws, _ = net._workspace(dev, batch, cpc)
    n = ctypes.c_int32()
    names = (ctypes.c_char_p * 64)()
    ms = (ctypes.c_float * 64)()
    cnt = (ctypes.c_int32 * 64)()
    y = torch.empty(batch, 2, HOP * cpc, device=dev)
    x = x_dev[..., :HOP * cpc + 64].contiguous()
    if x.shape[0] != batch:
        x = x[:1].expand(batch, -1, -1).contiguous()
    if emb.shape[0] != batch:
        emb = emb[:1].expand(batch, -1).contiguous()
    with torch.cuda.device(dev):
        _cabi.check(L.l2h_sep_profile(net._engine(), x.data_ptr(), x.shape[-1], emb.data_ptr(), st.buf.data_ptr(),
                                      y.data_ptr(), batch, cpc, ws.data_ptr(), ws.numel(), iters, names, ms, cnt,
                                      ctypes.byref(n), torch.cuda.current_stream(dev).cuda_stream))
    out = {}
    for i in range(n.value):
        out[names[i].decode()] = {"ms_total": ms[i] / iters, "ms_mean": ms[i] / max(1, cnt[i])}
    return out


if __name__ == "__main__":
    main()
