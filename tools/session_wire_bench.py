"""Streaming wire output (af_session_enable_wire) on the cfg5 shape: 1024 streams x 960-sample 48 kHz mono f32 ticks,
80 mels, VAD on.  Three legs, alternated tick by tick in one process:
  plain      the device-resident push exactly as bench.py's measure_cfg5 does it;
  wire_dev   the same push with the gated wire output (PCM16 + base64) to device rows;
  rings_host host-fed: af_session_push_rings from pinned capture rings, gated wire output to pinned host rows, then
             af_session_wire -- the loop of the app's processing task before send_audio.
Per leg: p50 / p99 / mean host time per tick (every push ends in a stream synchronise), kernels launched per tick
(af_kernel_launch_count) and bytes copied device-to-host per tick (computed from the tick's shapes), plus the device name
and power limit read through NVML in the same run.  Prints one JSON line.

    timeout 900 python tools/session_wire_bench.py [--ticks 500]
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
for p in (ROOT, os.path.join(ROOT, "audio-flow-rs_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402


def device_info(index: int = 0) -> dict:
    import pynvml
    pynvml.nvmlInit()
    try:
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        name = pynvml.nvmlDeviceGetName(h)
        return {"device": name.decode() if isinstance(name, bytes) else name,
                "power_limit_w": pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0}
    finally:
        pynvml.nvmlShutdown()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=500, help="timed ticks per leg (after 20 untimed ones)")
    ap.add_argument("--streams", type=int, default=1024)
    args = ap.parse_args()
    import torch
    import audioflow as af
    from audioflow import synth

    S, tick, warm = args.streams, 960, 20
    af.init(0)
    L = af.load_library()
    dev = torch.device("cuda:0")
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=True))
    x = synth.torch_batch(S, 2.0, 48000, 1, dev, seed=0)
    x_host = x.cpu().numpy()
    pcm = torch.empty((S, 512), device=dev)
    lm = torch.empty((S, 8 * 80), device=dev)
    vad = torch.zeros((S, 16), device=dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 512, lm.data_ptr(), 8 * 80, vad.data_ptr(), 16, None, 0, None)

    def session(wire_mem=None):
        h = C.c_void_p()
        af._check(L.af_session_create(pipe._h, S, 48000, 1, af.AF_FMT_F32, tick, C.byref(h)))
        if wire_mem is not None:
            cfg = af.WireConfigC(1, 1, 1, wire_mem)
            af._check(L.af_session_enable_wire(h, C.byref(cfg)))
        return h

    legs = {"plain": session(), "wire_dev": session(af.AF_MEM_DEVICE), "rings_host": session(af.AF_MEM_HOST)}
    rings = [af.RingBuffer(4 * tick) for _ in range(S)]
    ring_arr = (C.c_void_p * S)(*[r._h for r in rings])
    ticks = (af.WireTickC * S)()
    pp, ps, bp, bs, ff = C.c_void_p(), C.c_uint64(), C.c_void_p(), C.c_uint64(), C.c_uint64()
    nv = np.zeros(S, np.uint32)
    u32p = C.POINTER(C.c_uint32)
    tick_rec = C.sizeof(af.WireTickC)
    lat = {k: [] for k in legs}
    launches = {k: 0 for k in legs}
    d2h = {k: 0 for k in legs}
    torch.cuda.synchronize()
    names = list(legs)
    for t in range(warm + args.ticks):
        off = (t % 100) * tick
        for i in range(S):                                       # the capture callback's writes: not timed
            rings[i].write(x_host[i, off:off + tick])
        order = names[t % 3:] + names[:t % 3]                    # alternate which leg goes first
        for leg in order:
            h = legs[leg]
            l0 = L.af_kernel_launch_count()
            t0 = time.perf_counter()
            if leg == "rings_host":
                af._check(L.af_session_push_rings(h, ring_arr, tick, None, None, None, nv.ctypes.data_as(u32p)))
                af._check(L.af_session_wire(h, C.byref(pp), C.byref(ps), C.byref(bp), C.byref(bs), ticks, C.byref(ff)))
            else:
                af._check(L.af_session_push(h, x.data_ptr() + off * 4, x.shape[1], tick, af.AF_MEM_DEVICE, C.byref(o),
                                            None, None, None))
            dt = time.perf_counter() - t0
            if t >= warm:
                lat[leg].append(dt)
                launches[leg] += L.af_kernel_launch_count() - l0
                if leg == "wire_dev":
                    d2h[leg] += S * tick_rec                          # the tick records
                elif leg == "rings_host":
                    n = int(nv[0]) * 160                              # gated payload bound: the tick's frames x hop
                    d2h[leg] += S * (tick_rec + 2 * n + (L.af_pcm16_base64_len(n) if n else 0))
    for h in legs.values():
        L.af_session_destroy(h)
    res = {"tool": "session_wire_bench", "streams": S, "tick_samples": tick, "rate": 48000, "n_mels": 80, "vad": True,
           "ticks": args.ticks, "warmup_ticks": warm}
    for leg, v in lat.items():
        a = np.array(v) * 1e3
        res[leg] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "mean_ms": float(a.mean()),
                    "kernel_launches_per_tick": launches[leg] / args.ticks, "d2h_bytes_per_tick": d2h[leg] / args.ticks}
    res.update(device_info(0))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
