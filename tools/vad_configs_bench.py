"""Per-stream VAD configurations: what the records cost the scan kernels (batches) and the session tick.

Batch legs, alternated round by round in one process, device batches with device outputs:
  none          no records: the pipeline's configuration (the parent's code path);
  same          every stream the same configuration, not the pipeline's (a table of identical records);
  distinct8     8 distinct configurations cycled over the streams, all on the parallel scan;
  distinct8_seq the same with one stream at smoothing 0.05 (the sequential kernel follows the parallel one for it).
Shapes: cfg2 (256 x 30 s at 48 kHz mono, 80 mels, VAD on) and an hour (8 x 1 h at 48 kHz mono, VAD on, no mels: the
many-CTA scan).  Per leg: device time of the scan kernels (af_vad_scan*, af_vad_long_*) from torch.profiler, the device
time of the whole af_batch_run from CUDA events, and kernel launches per run.

Session legs (cfg5 shape: 1024 x 20 ms at 48 kHz mono, 80 mels, VAD on, device rows), alternated tick by tick:
  untouched     no configuration ever set;
  set_once      4 distinct configurations set once before the timed ticks;
  churn         1 % of the streams get a new configuration before every tick (the setter call is timed with the push).
Per leg: p50 / p99 / mean host time per tick (every push ends in a stream synchronise), launches per tick, and the bytes of
records uploaded per tick (counted from the ranges set since the previous push).  The device name and power limit are
read through NVML in the same run.  Prints one JSON line.

    timeout 900 python tools/vad_configs_bench.py [--runs 20] [--ticks 500]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
for p in (ROOT, os.path.join(ROOT, "audio-flow-rs_b200"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

from session_wire_bench import device_info  # noqa: E402

REC_BYTES = 32                    # sizeof(ScanRec): VadParams + warm-up + path flag
SCAN_KERNELS = ("af_vad_scan", "af_vad_long")


def _configs(af):
    V = af.VadConfig
    eight = [V(-45.0, 0.3, 15, 3), V(-50.0, 0.2, 10, 3), V(-55.0, 0.5, 20, 2), V(-40.0, 0.3, 15, 5),
             V(-50.0, 0.3, 5, 1), V(-60.0, 0.4, 40, 10), V(-35.0, 0.25, 15, 0), V(-48.0, 0.6, 12, 4)]
    return {"none": "unset", "same": [V(-45.0, 0.3, 15, 3)], "distinct8": eight,
            "distinct8_seq": [V(-50.0, 0.05, 15, 3)] + eight[1:]}


def bench_batch(af, torch, name, S, seconds, n_mels, runs):
    from audioflow import synth
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda:0")
    x = synth.torch_batch(S, seconds, 48000, 1, dev, seed=1)
    pipe = af.Pipeline(af.pipeline_config(n_mels=n_mels, vad_enable=True))
    legs = _configs(af)
    batches = {}
    for leg, cfgs in legs.items():
        b = pipe.batch([(x[i].data_ptr(), x.shape[1], 48000, 1, af.AF_FMT_F32) for i in range(S)], af.AF_MEM_DEVICE)
        if cfgs != "unset":
            b.set_vad_configs([cfgs[i % len(cfgs)] for i in range(S)])
        batches[leg] = b
    b0 = batches["none"]
    pcm = torch.empty((S, b0.pcm_stride), device=dev)
    lm = torch.empty((S, max(b0.logmel_stride, 4)), device=dev)
    vad = torch.zeros((S, b0.vad_stride), device=dev, dtype=torch.uint8)
    o = b0.outputs_struct(pcm.data_ptr(), b0.pcm_stride, lm.data_ptr() if n_mels else 0, b0.logmel_stride,
                          vad.data_ptr(), b0.vad_stride)
    st = torch.cuda.Stream()
    L = af.load_library()
    for b in batches.values():                                     # warm-up: modules, scratch
        b.run_device(o, st.cuda_stream)
    torch.cuda.synchronize()
    names = list(legs)
    run_ms = {k: [] for k in names}
    scan_us = {k: 0.0 for k in names}
    launches = {k: 0 for k in names}
    for r in range(runs):
        order = names[r % len(names):] + names[:r % len(names)]
        for leg in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = L.af_kernel_launch_count()
            e0.record(st)
            batches[leg].run_device(o, st.cuda_stream)
            e1.record(st)
            e1.synchronize()
            launches[leg] += L.af_kernel_launch_count() - l0
            run_ms[leg].append(e0.elapsed_time(e1))
    n_prof = max(runs // 4, 3)
    for leg in names:                                              # the scan kernels' device time, a profiler run per leg
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_prof):
                batches[leg].run_device(o, st.cuda_stream)
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if any(k in ev.key for k in SCAN_KERNELS):
                scan_us[leg] += ev.device_time_total / n_prof
    out = {"shape": name, "streams": S, "seconds": seconds, "n_mels": n_mels, "runs": runs}
    for leg in names:
        a = np.array(run_ms[leg])
        out[leg] = {"scan_us": round(scan_us[leg], 2), "run_p50_ms": float(np.percentile(a, 50)),
                    "run_mean_ms": float(a.mean()), "kernel_launches_per_run": launches[leg] / runs}
    del batches, x, pcm, lm, vad
    torch.cuda.empty_cache()
    return out


def bench_session(af, torch, ticks):
    from audioflow import synth
    dev = torch.device("cuda:0")
    S, tick, warm = 1024, 960, 20
    L = af.load_library()
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=True))
    x = synth.torch_batch(S, 4.0, 48000, 1, dev, seed=2)
    W = x.shape[1]
    pcm = torch.empty((S, 512), device=dev)
    lm = torch.empty((S, 8 * 80), device=dev)
    vad = torch.zeros((S, 16), device=dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 512, lm.data_ptr(), 8 * 80, vad.data_ptr(), 16, None, 0, None)
    names = ["untouched", "set_once", "churn"]
    ses = {k: af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for k in names}
    four = _configs(af)["distinct8"][:4]
    ses["set_once"].set_vad_configs(range(S), [four[i % 4] for i in range(S)])
    pool = _configs(af)["distinct8"]
    rng = np.random.default_rng(0)
    lat = {k: [] for k in names}
    launches = {k: 0 for k in names}
    h2d = {k: 0 for k in names}
    pending = {k: (S, 0) for k in names}                            # range of records set since the last push
    pending["set_once"] = (0, S)
    torch.cuda.synchronize()
    for t in range(warm + ticks):
        ptr = x.data_ptr() + ((t % 150) * tick) * 4
        ids = rng.choice(S, S // 100, replace=False)
        new = [pool[int(i)] for i in rng.integers(0, len(pool), ids.size)]
        order = names[t % len(names):] + names[:t % len(names)]
        for leg in order:
            s = ses[leg]
            l0 = L.af_kernel_launch_count()
            t0 = time.perf_counter()
            if leg == "churn":
                s.set_vad_configs(ids, new)
            af._check(L.af_session_push(s._h, ptr, W, tick, af.AF_MEM_DEVICE, C.byref(o), None, None, None))
            dt = time.perf_counter() - t0
            lo, hi = pending[leg]
            if leg == "churn":
                lo, hi = min(lo, int(ids.min())), max(hi, int(ids.max()) + 1)
                if t == 0:
                    lo, hi = 0, S                                   # the first upload takes the whole table
            uploaded = max(hi - lo, 0) * REC_BYTES if leg != "untouched" else 0
            pending[leg] = (S, 0)
            if t < warm:
                continue
            lat[leg].append(dt)
            launches[leg] += L.af_kernel_launch_count() - l0
            h2d[leg] += uploaded
    out = {"shape": "cfg5", "streams": S, "tick_samples": tick, "ticks": ticks, "warmup_ticks": warm,
           "churn_fraction_per_tick": 0.01}
    for leg in names:
        a = np.array(lat[leg]) * 1e6
        out[leg] = {"p50_us": float(np.percentile(a, 50)), "p99_us": float(np.percentile(a, 99)), "mean_us": float(a.mean()),
                    "kernel_launches_per_tick": launches[leg] / ticks, "record_h2d_bytes_per_tick": h2d[leg] / ticks}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=20, help="timed batch runs per leg")
    ap.add_argument("--ticks", type=int, default=500, help="timed session ticks per leg (after 20 untimed ones)")
    args = ap.parse_args()
    import torch
    import audioflow as af
    af.init(0)
    res = {"tool": "vad_configs_bench",
           "batch": [bench_batch(af, torch, "cfg2", 256, 30.0, 80, args.runs),
                     bench_batch(af, torch, "hour", 8, 3600.0, 0, max(args.runs // 2, 4))],
           "session": bench_session(af, torch, args.ticks)}
    res.update(device_info(0))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
