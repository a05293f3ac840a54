"""Polyphase resampling of batches (af_batch_set_resampler): what the anti-alias FIR costs against the cubic default.

Shapes, device batches with device outputs, 80 mels, VAD on:
  cfg2  256 x 30 s at 48 kHz mono f32;
  cfg3  4096 x 30 s, half 44.1 kHz and half 48 kHz mono f32 (interleaved in the batch).
Legs, alternated round by round in one process on one CUDA stream: cubic (the default path) and polyphase (the same
input, a second batch with the filter set).  Per leg the device time of the whole af_batch_run from CUDA events.  A
separate torch.profiler run per leg gives the device time of af_polyphase_fir_kernel and af_fused_kernel*.

The FIR's algorithmic bytes are the raw input read once plus the f32 rows written once (the stage halo, 60 of every 5436
samples at 48 kHz, is left out), and its FMAs are outputs x taps per output ((2L + 1) / q on average).  The FIR's HBM
bound is those bytes at 6544.3 GB/s, the copy bandwidth measured on the B200 (BASELINE.md).  The device name and power
limit are read through NVML in the same run.  Prints one JSON line.

    timeout 900 python tools/batch_polyphase_bench.py [--runs 10] [--shapes cfg2,cfg3]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
for p in (ROOT, os.path.join(ROOT, "audio-flow-rs_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from session_wire_bench import device_info  # noqa: E402

HBM_GBPS = 6544.3
FIR = "af_polyphase_fir_kernel"
FUSED = "af_fused_kernel"


def shape_streams(name):
    if name == "cfg2":
        return [(48000, 30.0)] * 256
    if name == "cfg3":
        return [(44100 if i % 2 else 48000, 30.0) for i in range(4096)]
    raise ValueError(name)


def fir_counts(af, rates, n_out):
    """(bytes, fmas) of the FIR over the streams: input read once, rows written once; outputs x mean taps."""
    b, f = 0, 0
    for (rate, sec), n in zip(rates, n_out):
        h, p, q = af.debug_polyphase_filter(rate)
        b += int(rate * sec) * 4 + int(n) * 4
        f += int(n) * (1 if p == q == 1 else len(h) / q)
    return b, f


def bench_shape(af, torch, name, runs):
    from audioflow import synth
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda:0")
    rates = shape_streams(name)
    S = len(rates)
    by_rate = {}
    for r in sorted(set(r for r, _ in rates)):
        idx = [i for i, (rr, _) in enumerate(rates) if rr == r]
        by_rate[r] = (idx, synth.torch_batch(len(idx), rates[idx[0]][1], r, 1, dev, seed=r))
    descs = [None] * S
    for r, (idx, x) in by_rate.items():
        for j, i in enumerate(idx):
            descs[i] = (x[j].data_ptr(), x.shape[1], r, 1, af.AF_FMT_F32)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=True))
    legs = {"cubic": pipe.batch(descs, af.AF_MEM_DEVICE), "polyphase": pipe.batch(descs, af.AF_MEM_DEVICE)}
    legs["polyphase"].set_resampler("polyphase")
    b0 = legs["cubic"]
    pcm = torch.empty((S, b0.pcm_stride), device=dev)
    lm = torch.empty((S, b0.logmel_stride), device=dev)
    vad = torch.zeros((S, b0.vad_stride), device=dev, dtype=torch.uint8)
    o = b0.outputs_struct(pcm.data_ptr(), b0.pcm_stride, lm.data_ptr(), b0.logmel_stride, vad.data_ptr(), b0.vad_stride)
    st = torch.cuda.Stream()
    L = af.load_library()
    for b in legs.values():                                         # warm-up: modules, scratch
        b.run_device(o, st.cuda_stream)
    torch.cuda.synchronize()
    names = list(legs)
    run_ms = {k: [] for k in names}
    launches = {k: 0 for k in names}
    for r in range(runs):
        for leg in (names if r % 2 == 0 else names[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = L.af_kernel_launch_count()
            e0.record(st)
            legs[leg].run_device(o, st.cuda_stream)
            e1.record(st)
            e1.synchronize()
            launches[leg] += L.af_kernel_launch_count() - l0
            run_ms[leg].append(e0.elapsed_time(e1))
    n_prof = max(runs // 2, 3)
    kern = {k: {} for k in names}
    for leg in names:                                               # kernel device times, a profiler run per leg
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_prof):
                legs[leg].run_device(o, st.cuda_stream)
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            for k in (FIR, FUSED):
                if k in ev.key:
                    kern[leg][k] = kern[leg].get(k, 0.0) + ev.device_time_total / n_prof
    fb, ff = fir_counts(af, rates, b0.n_out[:S])
    out = {"shape": name, "streams": S, "runs": runs, "fir_bytes": fb, "fir_fmas": ff,
           "fir_hbm_bound_us": round(fb / (HBM_GBPS * 1e9) * 1e6, 2)}
    for leg in names:
        a = np.array(run_ms[leg])
        out[leg] = {"run_p50_ms": round(float(np.percentile(a, 50)), 4), "run_mean_ms": round(float(a.mean()), 4),
                    "run_min_ms": round(float(a.min()), 4), "kernel_launches_per_run": launches[leg] / runs,
                    "kernel_us": {k: round(v, 2) for k, v in kern[leg].items()}}
    fir_us = kern["polyphase"].get(FIR, 0.0)
    if fir_us > 0:
        out["fir_gbps"] = round(fb / (fir_us * 1e-6) / 1e9, 1)
        out["fir_fraction_of_hbm_bound"] = round(out["fir_hbm_bound_us"] / fir_us, 3)
        out["fir_gfma_per_s"] = round(ff / (fir_us * 1e-6) / 1e9, 1)
    del legs, by_rate, pcm, lm, vad
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=10, help="timed runs per leg")
    ap.add_argument("--shapes", default="cfg2,cfg3")
    args = ap.parse_args()
    import torch
    import audioflow as af
    af.init(0)
    res = {"device_info": device_info(0), "hbm_gbps": HBM_GBPS}
    for s in args.shapes.split(","):
        res[s] = bench_shape(af, torch, s, args.runs)
        print(json.dumps(res[s]), file=sys.stderr, flush=True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
