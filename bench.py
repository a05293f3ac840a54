#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 audio hot path (BASELINE.json metric:
audio-seconds processed per second; HBM GB/s vs measured peak; CPU path timed beside it).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the fused pipeline (downmix -> resample -> STFT -> log-mel, PCM and
log-mel written) over one batch of BASELINE config 2 per GPU: 256 x 30 s 48 kHz mono f32 streams.
N > 1 shards independent streams across ranks (256 per rank, weak scaling).  cfg2 has no VAD, hence
nothing to exchange: the main line runs no collective.  Where there IS an exchange step -- the gather
of per-stream VAD states (`with_vad`, `cfg3`) -- it runs inside libaudioflow_gpu (NCCL, side stream);
torch.distributed only ships the 128-byte NCCL id and reduces the timings.

Extra keys of the line: `with_vad` (cfg2 + VAD + gather), `cfg3` (4096 x 30 s mixed 44.1/48 kHz,
stream-sharded over the N GPUs, strong scaling, with and without the gather), at N = 1 also `cfg4`
(1 h stereo, 128 mel, VAD + segmentation + gated output), `cfg5` (1024 x 20 ms ticks), `sustained`
(200 steps), `e2e_variants` (i16 in / PCM16 out / features only) and `parity` (measured log-mel error).
PyTorch is used only for device memory, streams/events and torch.distributed.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [os.path.join(ROOT, "audio-flow-rs_b200"), os.path.join(ROOT, "oracle")]
sys.dont_write_bytecode = True      # the bench writes nothing into the tree it runs from (which may be read-only)

STREAMS_PER_GPU = 256
SECONDS = 30.0
RATE = 48000
N_MELS = 80
# SURVEY.md 8(d): algorithmic bytes per audio-second = R_in*C*b_in + 16000*4 (PCM) + 100*M*4 (log-mel)
BYTES_PER_AUDIO_S = RATE * 1 * 4 + 16000 * 4 + 100 * N_MELS * 4          # 288000 (VAD off)
BYTES_PER_AUDIO_S_VAD = BYTES_PER_AUDIO_S + 100                          # + u8 VAD state per frame
WORKLOAD = "cfg2: 256 x 30 s 48 kHz mono f32 streams per GPU -> 16 kHz PCM + 25/10 ms STFT + 80-bin log-mel"
PRE_MS = float(os.environ.get("AF_BENCH_PRE_MS", "50"))   # untimed load in front of a timed window (0 under ncu: fixed launch counts)
DUMP_STREAMS = 16     # --dump-outputs: whole streams of a fixed, seeded sample of the batch (16 x 2.88 MB; all 256 are 737 MB)


def config_dict(world: int, variant: str = "auto") -> dict:
    """The `config` object of the JSON line -- identical for the GPU arm and the reference arm."""
    return {"workload": WORKLOAD, "streams_per_gpu": STREAMS_PER_GPU, "seconds": SECONDS, "sample_rate": RATE,
            "n_mels": N_MELS, "vad": False, "parallelism": f"stream-sharded x{world}", "bytes_per_audio_s": BYTES_PER_AUDIO_S,
            "l2": "inputs (1.47 GB per GPU) larger than L2; no explicit flush", "kernel_variant": variant}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = str(e)

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                     0x4: "sw_power_cap", 0x80: "hw_power_brake_slowdown"}
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while not self._stop_evt.is_set():
            self.sample()
            self._stop_evt.wait(0.005)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def pipe_stats_clear():
    import audioflow as af
    buf = (C.c_uint64 * 32)()
    af._check(af.load_library().af_debug_pipe_stats(buf))


def pipe_stats_print():
    """Per-role wait / work cycles of the fused kernel since the last clear (library built with `make STATS=1`)."""
    import audioflow as af
    buf = (C.c_uint64 * 32)()
    af._check(af.load_library().af_debug_pipe_stats(buf))
    names = {"fft": ("wait y_full", "wait p_empty"), "mel": ("wait p_full",),
             "vad": ("wait stage_empty", "wait y_full", "issue_fill"),
             "resample": ("wait y_empty", "wait stage_full", "tile setup", "carry+sync", "resample loops")}
    for r, (role, waits) in enumerate(names.items()):
        tot = max(int(buf[8 * r]), 1)
        print(f"[pipe-stats] {role:9s} warp-cycles {tot:.3e}  " +
              "  ".join(f"{w}: {100.0 * int(buf[8 * r + 1 + i]) / tot:5.1f}%" for i, w in enumerate(waits)), file=sys.stderr)


# ---------------------------------------------------------------------------------------------
# CPU legs (the oracle port of the reference path; the only place bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------
PORT_NOTE = ("oracle/oracle.c port of the reference CPU path (the reference is Rust and cannot be built here): to_mono "
             "(capture.rs:30-42) + BatchResampler over rubato FastFixedIn cubic (resampler.rs:132-166) = `reference_stages`; "
             "the f32 STFT/log-mel of the spec (`spec_stages`) is NOT reference code -- the reference has none")


def _cpu_inputs(n_streams, n):
    from audioflow import synth
    rng = np.random.default_rng(0)
    base = synth.stream(0, 4.0, RATE, 1)
    reps = int(np.ceil(n / len(base)))
    return [np.ascontiguousarray(np.tile(np.roll(base, int(rng.integers(0, len(base)))), reps)[:n]) for _ in range(min(n_streams, 8))]


def cpu_pipeline_rate(n_streams: int, seconds: float, stages: str = "all", repeats: int = 1, threads: int | None = None):
    """Times the CPU restatement of the path on n_streams synthetic streams of the bench shape spread over the host
    threads.  stages: "all" (cfg2: downmix + resample + f32 STFT/log-mel), "reference" (downmix + BatchResampler only --
    the stages the reference has code for), "spec" (the f32 STFT/log-mel alone, on already resampled PCM).
    Returns (audio_s_per_s, threads, best_seconds)."""
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    L = oracle.lib()
    cores = threads or os.cpu_count() or 1
    n = int(seconds * RATE)
    xs = _cpu_inputs(n_streams, n)
    plan = oracle.FeatPlan(oracle.default_feat_config(N_MELS))
    cap = L.orc_resample_max_output(RATE, 16000, n)
    fp = C.POINTER(C.c_float)
    pcm_ready = None
    if stages == "spec":
        pcm_ready = [oracle.resample_stream(x, RATE) for x in xs]

    def work(i):
        x = xs[i % len(xs)]
        T = cap // 160 + 1
        lm = np.empty(T * N_MELS, np.float32)
        if stages == "spec":
            y = pcm_ready[i % len(xs)]
            return L.orc_logmel_f32(plan._h, y.ctypes.data_as(fp), len(y), lm.ctypes.data_as(fp))
        mono = np.empty(n, np.float32)
        pcm = np.empty(cap, np.float32)
        vad = np.empty(T, np.uint8)
        nf = C.c_size_t(0)
        L.orc_pipeline_stream(x.ctypes.data_as(fp), n, 1, RATE, plan._h if stages == "all" else None, None, 400, 160,
                              mono.ctypes.data_as(fp), pcm.ctypes.data_as(fp), cap,
                              lm.ctypes.data_as(fp) if stages == "all" else None, vad.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(nf))
        return nf.value

    best = None
    with ThreadPoolExecutor(max_workers=cores) as ex:
        for _ in range(repeats):
            t0 = time.perf_counter()
            list(ex.map(work, range(n_streams)))
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    return n_streams * seconds / best, cores, best


def cpu_cfg1_single_thread():
    """BASELINE config 1 -- "the reference path": ONE 10 s 48 kHz stereo f32 clip -> mono 16 kHz + VAD on 20 ms frames,
    single-threaded.  `port`: the stages with caller-provided buffers; `reference_shaped`: the same arithmetic driven as the
    reference's processing loop would (100 ms reads) WITH the Vec allocations / copies / drain the Rust code performs."""
    import oracle
    from audioflow import synth
    L = oracle.lib()
    x = synth.stream(1, 10.0, 48000, 2)
    fp, u8p = C.POINTER(C.c_float), C.POINTER(C.c_uint8)
    n = len(x)
    mono = np.empty(n // 2 + 1, np.float32)
    cap = L.orc_resample_max_output(48000, 16000, n // 2)
    pcm = np.empty(cap, np.float32)
    vad = np.empty(cap // 320 + 2, np.uint8)
    nf = C.c_size_t(0)
    vc = oracle.default_vad_config()

    def port():
        L.orc_pipeline_stream(x.ctypes.data_as(fp), n, 2, 48000, None, C.byref(vc), 320, 320, mono.ctypes.data_as(fp),
                              pcm.ctypes.data_as(fp), cap, None, vad.ctypes.data_as(u8p), C.byref(nf))

    def shaped():
        L.orc_pipeline_stream_shaped(x.ctypes.data_as(fp), n, 2, 48000, 4800, C.byref(vc), 320, pcm.ctypes.data_as(fp), cap,
                                     vad.ctypes.data_as(u8p), C.byref(nf))

    out = {}
    for name, fn in (("port", port), ("reference_shaped", shaped)):
        fn()
        best = min(_t(fn) for _ in range(5))
        out[name] = {"audio_s_per_s": 10.0 / best, "ms": 1e3 * best}
    out["config"] = "cfg1: 1 x 10 s 48 kHz stereo f32 -> mono 16 kHz (BatchResampler) + VAD on 20 ms frames, 1 thread, best of 5"
    return out


def _t(fn):
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference is Rust and cannot be
    built in this image (no toolchain, rubato sources absent), so this is the oracle PORT of it, timed with all host
    threads on the SAME config: every step is one whole cfg2 batch (256 x 30 s)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import oracle
    oracle.lib()
    for _ in range(args.warmup):
        cpu_pipeline_rate(16, 5.0)
    t_total, units = 0.0, 0.0
    cores = os.cpu_count() or 1
    for _ in range(args.steps):
        rate, cores, dt = cpu_pipeline_rate(STREAMS_PER_GPU, SECONDS)
        t_total += dt
        units += STREAMS_PER_GPU * SECONDS
    value = units / t_total
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.gpus, args.variant),
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": cores, "kind": "port",
                         "sample": f"every step = the whole cfg2 batch of ONE GPU ({STREAMS_PER_GPU} x {SECONDS:.0f} s) on {cores} host threads, {args.steps} steps; " + PORT_NOTE},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------
# GPU side
# ---------------------------------------------------------------------------------------------
class Env:
    """What every measurement needs: torch, the library, rank / world, the torch stream the library enqueues on."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import audioflow as af
        from audioflow import synth
        self.torch, self.dist, self.af, self.synth, self.args = torch, dist, af, synth, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (libaudioflow_gpu has no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", rank=self.rank, world_size=self.world, device_id=self.dev)
        af.init(self.local_rank)
        af.set_kernel_variant(args.variant)
        self.L = af.load_library()
        # a stream of our own (torch's default is the legacy NULL stream, which the C ABI reads as "the library's own"): torch
        # ops, the events of the timed regions and -- through af_set_stream -- everything the library enqueues share it
        self.stream = torch.cuda.Stream(device=self.dev)
        torch.cuda.set_stream(self.stream)
        assert self.stream.cuda_stream != 0
        af._check(self.L.af_set_stream(self.stream.cuda_stream))
        if self.world > 1:
            # the library's own communicator (ncclCommInitRank inside libaudioflow_gpu); torch.distributed only ships the id
            uid = torch.zeros(128, dtype=torch.uint8, device=self.dev)
            if self.rank == 0:
                uid.copy_(torch.tensor(list(af.comm_unique_id()), dtype=torch.uint8))
            dist.broadcast(uid, 0)
            af.comm_init_rank(self.world, self.rank, bytes(uid.cpu().tolist()))

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float):
        if self.world == 1:
            return v, [v]
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        allt = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(allt, t)
        vals = [float(x.item()) for x in allt]
        return max(vals), vals

    def timed(self, step, steps: int, warmup: int, clocks: bool = False, finish=None):
        """W untimed warm-up steps; barrier + synchronize; ~PRE_MS of untimed load so that the window does not start on a GPU
        that idled through the barrier; EXACTLY `steps` steps between two CUDA events on the launching stream;
        synchronize + barrier.  Returns (ms of the timed steps = max over ranks, per-rank ms, launches, clocks)."""
        torch, af = self.torch, self.af
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(self.stream)
        for _ in range(max(warmup, 1)):
            step()
        w1.record(self.stream)
        torch.cuda.synchronize()
        est, _ = self.max_over_ranks(max(w0.elapsed_time(w1) / max(warmup, 1), 1e-3))   # (every rank must run the SAME number of steps:
        n_pre = int(min(max(math.ceil(PRE_MS / est), 1), 5000))                          #  a step may hold a collective)
        self.barrier()
        sampler = ClockSampler(self.local_rank) if clocks else None
        for _ in range(n_pre):
            step()
        l0 = af.kernel_launch_count()
        e0.record(self.stream)
        for _ in range(steps):
            step()
        if finish is not None:
            finish()                      # e.g. order the stream after the last gather: the region ends when the results exist
        e1.record(self.stream)
        launches = af.kernel_launch_count() - l0
        if sampler:
            sampler.sample()
            sampler.start()
        torch.cuda.synchronize()
        if sampler:
            sampler.stop()
        self.barrier()
        ms = e0.elapsed_time(e1)
        ms_max, per_rank = self.max_over_ranks(ms)
        return ms_max, [round(v / steps, 4) for v in per_rank], launches, (sampler.summary() if sampler else None)


def dump_outputs(out_dir: str, b, pcm, lm):
    """What a caller of the timed cfg2 step holds after its last step: the 16 kHz PCM [k, n_out] and the log-mel
    [k, T, N_MELS] of DUMP_STREAMS streams picked with a fixed seed (sorted batch rows), as float32 .npy files.  The inputs
    are seeded too, so two builds of the library run with the same arguments can be compared output for output."""
    import torch
    rows = np.sort(np.random.default_rng(0).choice(STREAMS_PER_GPU, DUMP_STREAMS, replace=False))
    n_out, T = int(b.n_out[0]), int(b.n_feat[0])          # every stream of the batch has the same length
    idx = torch.as_tensor(rows, device=pcm.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pcm.npy"), pcm[idx, :n_out].cpu().numpy())
    np.save(os.path.join(out_dir, "logmel.npy"), lm[idx, :T * N_MELS].reshape(len(rows), T, N_MELS).cpu().numpy())


def measure_cfg2(env: Env, steps: int, warmup: int):
    """The contract line: cfg2 per GPU, VAD off, no collective; then the same with the VAD on and -- at N > 1 -- the
    gather of the VAD states inside the library."""
    af, torch, args = env.af, env.torch, env.args
    S, n = STREAMS_PER_GPU, int(SECONDS * RATE)
    x = env.synth.torch_batch(S, SECONDS, RATE, 1, env.dev, seed=env.rank)             # resident in HBM before timing
    descs = [(x[i].data_ptr(), n, RATE, 1, af.AF_FMT_F32) for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=N_MELS, vad_enable=False))
    b = pipe.batch(descs, af.AF_MEM_DEVICE)
    pcm = torch.empty((S, b.pcm_stride), device=env.dev)
    lm = torch.empty((S, b.logmel_stride), device=env.dev)
    o = b.outputs_struct(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride)
    st = env.stream.cuda_stream

    def step():
        b.run_device(o, st)

    if args.pipe_stats:
        pipe_stats_clear()
    ms, per_rank, launches, clocks = env.timed(step, steps, warmup, clocks=True)
    if args.pipe_stats:
        pipe_stats_print()
    if args.dump_outputs and env.rank == 0:
        dump_outputs(args.dump_outputs, b, pcm, lm)      # before the runs below reuse pcm / lm
    res = {"ms_per_step": ms / steps, "per_rank": per_rank, "launches": launches, "clocks": clocks, "x": x, "pipe": pipe,
           "lm": lm, "batch": b}
    if not args.quick:
        ms200, _, _, _ = env.timed(step, 200, 3)
        res["sustained_ms"] = ms200 / 200

    # ---- VAD on: fused kernel with the energy chains + scan kernel; N > 1: + the NCCL gather of the states ----
    pipe_v = af.Pipeline(af.pipeline_config(n_mels=N_MELS, vad_enable=True))
    geo = [(descs[i % S][0] if r == env.rank else 0, n, RATE, 1, af.AF_FMT_F32) for r in range(env.world) for i in range(S)]
    sb = af.ShardedBatch(pipe_v, geo, af.AF_MEM_DEVICE)
    lb = sb.local(env.rank)
    outs = af.ShardedOutputsC()
    outs.shard[env.rank] = af.OutputsC(pcm.data_ptr(), lb.pcm_stride, lm.data_ptr(), lb.logmel_stride, None, 0, None, 0, None)

    def step_v():
        sb.run(outs, gather=True, wait=False)

    if args.pipe_stats:
        env.timed(step_v, 2, 1)
        pipe_stats_clear()
    steps_v = max(steps // 2, 3)
    ms_v, per_rank_v, launches_v, _ = env.timed(step_v, steps_v, warmup, finish=sb.join)
    if args.pipe_stats:
        print("[pipe-stats] --- with the VAD on ---", file=sys.stderr)
        pipe_stats_print()
    gather_ms = sb.gather_ms(env.rank) if env.world > 1 else 0.0
    gmax, _ = env.max_over_ranks(gather_ms)
    res["with_vad"] = {"value": env.world * S * SECONDS / (ms_v / steps_v * 1e-3), "ms_per_step": ms_v / steps_v,
                       "per_rank_ms_per_step": per_rank_v, "gpu_launches_per_step": launches_v / steps_v,
                       "hbm_gbs": BYTES_PER_AUDIO_S_VAD * S * SECONDS / (ms_v / steps_v * 1e-3) / 1e9,
                       "gather": ("one in-place ncclAllGather of the u8 VAD states per step inside libaudioflow_gpu, on a low-priority side "
                                  "stream; the scan kernel writes straight into the double-buffered gather buffer; the timed region ends "
                                  "after the last gather") if env.world > 1 else "none (1 GPU)",
                       "gather_ms": gmax, "gather_bytes_per_rank": int(S * lb.vad_stride)}
    if not args.quick:
        ms200, _, _, _ = env.timed(step_v, 200, 3, finish=sb.join)
        res["with_vad"]["sustained_ms_per_step"] = ms200 / 200
    del sb
    return res


def pcie_ceiling_ms(env: Env, h2d_bytes: int, d2h_bytes: int, reps: int = 3):
    """What the host link of THIS box gives for the same bytes: pinned H2D and D2H on two streams at once (every rank at the
    same time at N > 1).  The e2e leg cannot be faster than this."""
    torch = env.torch
    hin = torch.empty(max(h2d_bytes, 4) // 4, dtype=torch.float32).pin_memory()
    hout = torch.empty(max(d2h_bytes, 4) // 4, dtype=torch.float32).pin_memory()
    din, dout = torch.empty_like(hin, device=env.dev), torch.empty_like(hout, device=env.dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def both():
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s2):
            hout.copy_(dout, non_blocking=True)

    both()
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        both()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    dt, _ = env.max_over_ranks(dt)
    return 1e3 * dt


def measure_e2e(env: Env, x, pipe_f32, lm_dev, steps: int):
    """The reference-facing call with HOST (pinned) buffers: af_batch_run_host, H2D + D2H inside the timed region.  The main
    variant is the contract's (f32 in, f32 PCM + log-mel out); the others cut the bytes that cross the host link."""
    af, torch, L = env.af, env.torch, env.L
    S, n = STREAMS_PER_GPU, int(SECONDS * RATE)
    out = {}
    variants = [("f32_in__f32_pcm+logmel", "f32", dict(n_mels=N_MELS, vad_enable=False))]
    if not env.args.quick:
        variants += [("i16_in__pcm16+logmel", "i16", dict(n_mels=N_MELS, vad_enable=False, pcm16=True)),
                     ("i16_in__logmel_only", "i16", dict(n_mels=N_MELS, vad_enable=False, write_pcm=False))]
    for name, fmt, kw in variants:
        bps = 2 if fmt == "i16" else 4
        in_bytes = S * n * bps
        hp = C.c_void_p()
        af._check(L.af_host_alloc(C.byref(hp), in_bytes))
        if fmt == "i16":
            hin = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_int16)), shape=(S, n))
            hin[:] = torch.round(x * 32767.0).to(torch.int16).cpu().numpy()
        else:
            hin = np.ctypeslib.as_array(C.cast(hp, C.POINTER(C.c_float)), shape=(S, n))
            hin[:] = x.cpu().numpy()
        pipe = pipe_f32 if name.startswith("f32_in") else af.Pipeline(af.pipeline_config(**kw))
        hdescs = [(hin[i].ctypes.data, n, RATE, 1, af.AF_FMT_I16 if fmt == "i16" else af.AF_FMT_F32) for i in range(S)]
        hb = pipe.batch(hdescs, af.AF_MEM_HOST)
        want_pcm = kw.get("write_pcm", True)
        pcm_el = 2 if kw.get("pcm16") else 4
        pcm_bytes, lm_bytes = (S * hb.pcm_stride * pcm_el if want_pcm else 0), S * hb.logmel_stride * 4
        po, pl = C.c_void_p(), C.c_void_p()
        if want_pcm:
            af._check(L.af_host_alloc(C.byref(po), pcm_bytes))
        af._check(L.af_host_alloc(C.byref(pl), lm_bytes))
        ho = hb.outputs_struct(po.value if want_pcm else 0, hb.pcm_stride, pl.value, hb.logmel_stride)
        af._check(L.af_batch_run_host(hb._h, C.byref(ho)))            # warm-up
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            af._check(L.af_batch_run_host(hb._h, C.byref(ho)))        # blocking: returns when results are on the host
        dt = time.perf_counter() - t0
        dt, _ = env.max_over_ranks(dt)
        d2h = int(S * ((int(hb.n_out.max()) * pcm_el if want_pcm else 0) + int(hb.n_feat.max()) * N_MELS * 4))
        r = {"value": env.world * steps * S * SECONDS / dt, "unit": "audio-s/s", "h2d_bytes_per_step": int(in_bytes),
             "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * dt / steps}
        if name.startswith("f32_in"):
            # spot-check of the e2e result against the device-resident run
            lm_host = np.ctypeslib.as_array(C.cast(pl, C.POINTER(C.c_float)), shape=(S, hb.logmel_stride))
            T = int(hb.n_feat[0])
            if not np.array_equal(lm_host[3, :T * N_MELS], lm_dev[3, :T * N_MELS].cpu().numpy()):
                raise SystemExit("e2e result differs from the device-resident result")
        del hb
        L.af_host_free(hp); L.af_host_free(pl)
        if want_pcm:
            L.af_host_free(po)
        r["pcie_ceiling_ms"] = pcie_ceiling_ms(env, in_bytes, d2h)
        r["frac_of_pcie_ceiling"] = r["pcie_ceiling_ms"] / r["ms_per_step"]
        out[name] = r
    main = out.pop("f32_in__f32_pcm+logmel")
    main["note"] = ("af_batch_run_host: pinned host PCM in, PCM + log-mel back on the host; 3-slot H2D/compute/D2H overlap over ~32 MB "
                    "groups of streams; pcie_ceiling_ms = the same bytes as bare pinned copies, both directions at once, every rank at once")
    return main, out


def measure_cfg3(env: Env, steps: int, warmup: int):
    """BASELINE config 3: 4096 x 30 s mixed 44.1/48 kHz mono f32, full pipeline (PCM + 80 mel + VAD), sharded over the N GPUs by
    input bytes inside the library (strong scaling), with and without the gather of the VAD states."""
    af, torch = env.af, env.torch
    S_total = int(os.environ.get("AF_CFG3_STREAMS", "4096"))                # (experiments: fewer streams / a single rate)
    only = os.environ.get("AF_CFG3_RATE")
    rates = [int(only) if only else (44100 if i % 2 else 48000) for i in range(S_total)]
    geo = [(0, int(SECONDS * r), r, 1, af.AF_FMT_F32) for r in rates]
    lo, hi = af.shard_partition(geo, env.world)[env.rank]
    mine = list(range(lo, hi))
    x48 = env.synth.torch_batch(max(sum(1 for i in mine if rates[i] == 48000), 1), SECONDS, 48000, 1, env.dev, seed=2 * env.rank)
    x44 = env.synth.torch_batch(max(sum(1 for i in mine if rates[i] == 44100), 1), SECONDS, 44100, 1, env.dev, seed=2 * env.rank + 1)
    descs, i48, i44 = list(geo), 0, 0
    for i in mine:
        if rates[i] == 48000:
            descs[i] = (x48[i48].data_ptr(), x48.shape[1], 48000, 1, af.AF_FMT_F32); i48 += 1
        else:
            descs[i] = (x44[i44].data_ptr(), x44.shape[1], 44100, 1, af.AF_FMT_F32); i44 += 1
    pipe = af.Pipeline(af.pipeline_config(n_mels=N_MELS, vad_enable=True))
    sb = af.ShardedBatch(pipe, descs, af.AF_MEM_DEVICE)
    b = sb.local(env.rank)
    S = len(mine)
    pcm = torch.empty((S, b.pcm_stride), device=env.dev)
    lm = torch.empty((S, b.logmel_stride), device=env.dev)
    vad = torch.zeros((S, b.vad_stride), device=env.dev, dtype=torch.uint8)
    outs = af.ShardedOutputsC()
    outs.shard[env.rank] = af.OutputsC(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, vad.data_ptr(), b.vad_stride, None, 0, None)
    if env.args.pipe_stats:
        pipe_stats_clear()
    ms0, per_rank0, _, _ = env.timed(lambda: sb.run(outs, gather=False, wait=False), steps, warmup)
    if env.args.pipe_stats:
        pipe_stats_print()
    ms1, per_rank1, _, _ = env.timed(lambda: sb.run(outs, gather=True, wait=False), steps, warmup, finish=sb.join)
    gather_ms, _ = env.max_over_ranks(sb.gather_ms(env.rank) if env.world > 1 else 0.0)
    audio_s = S_total * SECONDS
    alg = sum((r * 4 + 16000 * 4 + 100 * N_MELS * 4 + 100) * SECONDS for r in rates)
    peak, _ = measured_peak_gbs()
    ms0s, ms1s = ms0 / steps, ms1 / steps
    r = {"workload": "cfg3: 4096 x 30 s mixed 44.1/48 kHz mono f32 -> PCM + 80-mel + VAD, stream-sharded by input bytes (af_sharded_batch)",
         "metric": "audio_seconds_per_second", "unit": "audio-s/s", "n_gpus": env.world, "scaling": "strong",
         "value": audio_s / (ms1s * 1e-3), "ms_per_step": ms1s, "per_rank_ms_per_step": per_rank1,
         "value_without_gather": audio_s / (ms0s * 1e-3), "ms_per_step_without_gather": ms0s,
         "gather": ("u8 VAD states of every stream to every GPU: one in-place ncclAllGather per step inside libaudioflow_gpu (side stream, "
                    "double-buffered, written by the scan kernel)") if env.world > 1 else "none (1 GPU)",
         "gather_ms": gather_ms, "gather_bytes_per_rank": int(S * b.vad_stride),
         "hbm_gbs_per_gpu": alg / env.world / (ms0s * 1e-3) / 1e9, "hbm_frac_per_gpu": alg / env.world / (ms0s * 1e-3) / 1e9 / peak,
         "steps": steps, "warmup": warmup, "data": "synthetic"}
    del sb
    return r


def measure_cfg4(env: Env, steps: int, warmup: int):
    """BASELINE config 4: one 1-hour 48 kHz stereo recording -> PCM + 128-mel + VAD + segmentation + gated (speech-only) output.
    A single stream does not shard: replicas only."""
    af, torch, L = env.af, env.torch, env.L
    sec, M = 3600.0, 128
    x = env.synth.torch_batch(1, sec, 48000, 2, env.dev, seed=env.rank)
    pipe = af.Pipeline(af.pipeline_config(n_mels=M, vad_enable=True))
    b = pipe.batch([(x[0].data_ptr(), x.shape[1], 48000, 2, af.AF_FMT_F32)], af.AF_MEM_DEVICE)
    pcm = torch.empty((1, b.pcm_stride), device=env.dev)
    lm = torch.empty((1, b.logmel_stride), device=env.dev)
    vad = torch.zeros((1, b.vad_stride), device=env.dev, dtype=torch.uint8)
    seg_cap = 65536
    seg = torch.zeros((1, seg_cap, 2), device=env.dev, dtype=torch.int32)
    nseg = torch.zeros(1, device=env.dev, dtype=torch.int32)
    nfr = torch.tensor(b.n_vad[:1].astype(np.int32), device=env.dev)
    nout = torch.tensor(b.n_out[:1].astype(np.int32), device=env.dev)
    g_pcm, g_lm = torch.empty_like(pcm), torch.empty_like(lm)
    g_off = torch.zeros((1, seg_cap + 1), device=env.dev, dtype=torch.int32)
    g_n = torch.zeros(1, device=env.dev, dtype=torch.int32)
    go = af.GateOutputsC(g_pcm.data_ptr(), b.pcm_stride, g_lm.data_ptr(), b.logmel_stride, g_off.data_ptr(), g_n.data_ptr())
    o = b.outputs_struct(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, vad.data_ptr(), b.vad_stride)
    st = env.stream.cuda_stream

    def step():
        b.run_device(o, st)
        L.af_vad_segments(vad.data_ptr(), b.vad_stride, nfr.data_ptr(), 1, seg.data_ptr(), seg_cap, nseg.data_ptr(), st)

    def step_gate():
        step()
        L.af_vad_gate(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, M, nout.data_ptr(), 160, seg.data_ptr(), seg_cap,
                      nseg.data_ptr(), 1, C.byref(go), st)

    if env.args.pipe_stats:
        pipe_stats_clear()
    ms, _, _, _ = env.timed(step, steps, warmup)
    if env.args.pipe_stats:
        pipe_stats_print()
    msg, _, _, _ = env.timed(step_gate, steps, warmup)
    alg = (48000 * 2 * 4 + 16000 * 4 + 100 * M * 4 + 100) * sec
    peak, _ = measured_peak_gbs()
    mss = ms / steps
    return {"workload": "cfg4: 1 x 3600 s 48 kHz stereo f32 -> PCM + 128-mel + VAD + segmentation (replicas only)",
            "metric": "audio_seconds_per_second", "unit": "audio-s/s", "n_gpus": env.world, "value": env.world * sec / (mss * 1e-3),
            "ms_per_step": mss, "segments": int(nseg[0]), "ms_per_step_with_gated_output": msg / steps,
            "gated_frames": int(g_n[0]), "frames": int(b.n_vad[0]),
            "hbm_gbs_per_gpu": alg / (mss * 1e-3) / 1e9, "hbm_frac_per_gpu": alg / (mss * 1e-3) / 1e9 / peak, "steps": steps,
            "warmup": warmup, "data": "synthetic"}


def measure_cfg5(env: Env, n_ticks: int):
    """BASELINE config 5: 1024 concurrent 20 ms-chunk 48 kHz mono streams, persistent state, latency bound."""
    af, torch, L = env.af, env.torch, env.L
    S, tick = 1024, 960
    pipe = af.Pipeline(af.pipeline_config(n_mels=N_MELS, vad_enable=True))
    h = C.c_void_p()
    af._check(L.af_session_create(pipe._h, S, 48000, 1, af.AF_FMT_F32, tick, C.byref(h)))
    x = env.synth.torch_batch(S, 2.0, 48000, 1, env.dev, seed=env.rank)
    pcm = torch.empty((S, 512), device=env.dev)
    lm = torch.empty((S, 8 * N_MELS), device=env.dev)
    vad = torch.zeros((S, 16), device=env.dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 512, lm.data_ptr(), 8 * N_MELS, vad.data_ptr(), 16, None, 0, None)
    torch.cuda.synchronize()
    lat = []
    for t in range(n_ticks + 20):
        off = (t % 100) * tick
        t0 = time.perf_counter()
        af._check(L.af_session_push(h, x.data_ptr() + off * 4, x.shape[1], tick, af.AF_MEM_DEVICE, C.byref(o), None, None, None))
        if t >= 20:
            lat.append(time.perf_counter() - t0)
    L.af_session_destroy(h)
    lat = np.array(lat) * 1e3
    return {"workload": "cfg5: 1024 x 20 ms ticks (960 samples @ 48 kHz mono f32), persistent state, PCM + 80-mel + VAD per tick",
            "metric": "tick_latency_ms", "p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)),
            "mean_ms": float(lat.mean()), "ticks": int(len(lat)), "n_gpus": env.world,
            "realtime_factor": 20.0 / float(np.percentile(lat, 99)),
            "max_realtime_streams_per_gpu": int(S * 20.0 / float(np.percentile(lat, 99))),
            "audio_seconds_per_second": env.world * S * 0.02 / (float(lat.mean()) * 1e-3), "data": "synthetic"}


def cpu_leg(env: Env, x, lm_dev, batch):
    """cpu_baseline (rank 0, N = 1): the oracle port timed on the box's host threads, split into the stages the reference has
    code for and the spec-defined ones, cfg1 single-threaded, and -- the oracle as the CHECKER -- the measured log-mel error of
    the GPU result of this run on two of its streams."""
    import oracle
    S = STREAMS_PER_GPU
    v, cores, dt = cpu_pipeline_rate(S, SECONDS, "all", repeats=3)
    v_ref, _, dt_ref = cpu_pipeline_rate(S, SECONDS, "reference", repeats=2)
    v_spec, _, dt_spec = cpu_pipeline_rate(S, SECONDS, "spec", repeats=2)
    cpu = {"value": v, "unit": "audio-s/s", "cores": cores, "kind": "port",
           "sample": f"all {S} streams x {SECONDS:.0f} s, best of 3 passes (all {cores} host threads, {dt:.2f} s wall per pass); " + PORT_NOTE,
           "reference_stages": {"value": v_ref, "unit": "audio-s/s", "what": "downmix + BatchResampler(all) + flush (capture.rs:30-42, resampler.rs:132-166)"},
           "spec_stages": {"value": v_spec, "unit": "audio-s/s", "what": "f32 Hann + 512-pt FFT + 80 mel + log on the resampled PCM: NOT reference code"},
           "cfg1_single_thread": cpu_cfg1_single_thread()}
    fc = oracle.default_feat_config(N_MELS)
    G, R = [], []
    for i in (3, 200):
        y = oracle.resample_stream(x[i].cpu().numpy(), RATE)
        ref = oracle.logmel(y, fc)
        T = ref.shape[0]
        G.append(lm_dev[i, :T * N_MELS].reshape(T, N_MELS).cpu().numpy().astype(np.float64)); R.append(ref.astype(np.float64))
    g, r = np.concatenate(G), np.concatenate(R)
    err = np.abs(g - r)
    dr_db = (r.max(axis=1, keepdims=True) - r) * (10.0 / np.log(10.0))
    over = err > 1e-4
    parity = {"what": "log-mel of THIS run (streams 3 and 200 of the cfg2 batch) against the f64 oracle; PCM / VAD are bit-exact (tests/)",
              "logmel_max_abs": float(err.max()), "frac_bins_over_1e-4": float(over.mean()),
              "rel_l2": float(np.sqrt((err ** 2).sum() / (r ** 2).sum())), "bins": int(err.size),
              "max_abs_within_50dB_of_frame_peak": float(err[dr_db <= 50.0].max()),
              "min_dB_below_frame_peak_of_bins_over_1e-4": float(dr_db[over].min()) if over.any() else None}
    return cpu, parity


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="contract keys only: no e2e variants, no cfg3/4/5, no 200-step lines")
    ap.add_argument("--variant", default="auto")
    ap.add_argument("--pipe-stats", action="store_true",
                    help="print the fused kernel's per-role wait cycles (needs AF_GPU_LIB=.../libaudioflow_gpu_stats.so)")
    ap.add_argument("--workload", default="all", choices=["all", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="all = the contract line (cfg2) carrying the other configs as keys; cfgN = that config's object alone")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed cfg2 steps, write the PCM and log-mel of their last step (rank 0, a fixed sample of "
                         f"{DUMP_STREAMS} streams) as DIR/pcm.npy and DIR/logmel.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload not in ("all", "cfg2")):
        ap.error("--dump-outputs writes the outputs of the cfg2 line: not with --impl reference or --workload cfg3/cfg4/cfg5")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    if args.impl == "reference":
        return run_reference_arm(args)

    env = Env(args)
    rank, world = env.rank, env.world
    if args.workload in ("cfg3", "cfg4", "cfg5"):
        r = {"cfg3": lambda: measure_cfg3(env, args.steps, args.warmup), "cfg4": lambda: measure_cfg4(env, args.steps, args.warmup),
             "cfg5": lambda: measure_cfg5(env, max(args.steps, 500))}[args.workload]()
        if rank == 0:
            print(json.dumps(r), flush=True)
        if world > 1:
            env.af.comm_shutdown()
            env.dist.destroy_process_group()
        return 0

    S = STREAMS_PER_GPU
    c2 = measure_cfg2(env, args.steps, args.warmup)
    ms_per_step = c2["ms_per_step"]
    value = world * S * SECONDS / (ms_per_step * 1e-3)

    # ---- roofline of the dominant kernel: with the VAD off a step IS one launch of af_fused_kernel ----
    peak, peak_src = measured_peak_gbs()
    alg_bytes = BYTES_PER_AUDIO_S * S * SECONDS
    achieved = alg_bytes / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic, traffic_src = tj.get("af_fused_kernel_bytes_per_launch"), tj.get("source")
    except Exception:
        pass

    e2e, e2e_variants = (None, None)
    if args.e2e_steps > 0:
        e2e, e2e_variants = measure_e2e(env, c2["x"], c2["pipe"], c2["lm"], args.e2e_steps)

    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, parity = cpu_leg(env, c2["x"], c2["lm"], c2["batch"])
    for k in ("x", "lm", "batch", "pipe"):
        c2.pop(k)
    env.torch.cuda.empty_cache()

    cfg3 = cfg4 = cfg5 = None
    if args.workload == "all" and not args.quick:
        cfg3 = measure_cfg3(env, min(args.steps, 10), 2)
        env.torch.cuda.empty_cache()
        if world == 1:
            cfg4 = measure_cfg4(env, min(args.steps, 20), 3)
            cfg5 = measure_cfg5(env, 500)

    if rank == 0:
        line = {
            "metric": "audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(world, args.variant),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "kernel": "af_fused_kernel", "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes},
            "cpu_baseline": cpu,
            "e2e": e2e, "per_rank_ms_per_step": c2["per_rank"] if world > 1 else None,
            "gpu_launches": int(c2["launches"]),
            "clocks": c2["clocks"],
            "timing": f"W warm-up steps, barrier, ~{PRE_MS:.0f} ms of untimed steps, then K steps between CUDA events on the launching stream, max over ranks; no collective in the main line (cfg2 has no VAD: nothing to exchange)",
            "with_vad": c2["with_vad"],
        }
        if "sustained_ms" in c2:
            line["sustained"] = {"steps": 200, "ms_per_step": c2["sustained_ms"], "value": world * S * SECONDS / (c2["sustained_ms"] * 1e-3),
                                 "roofline_frac": alg_bytes / (c2["sustained_ms"] * 1e-3) / 1e9 / peak}
        if e2e_variants:
            line["e2e_variants"] = e2e_variants
        if parity:
            line["parity"] = parity
        for k, v in (("cfg3", cfg3), ("cfg4", cfg4), ("cfg5", cfg5)):
            if v is not None:
                line[k] = v
        print(json.dumps(line), flush=True)
    if world > 1:
        env.af.comm_shutdown()
        env.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
