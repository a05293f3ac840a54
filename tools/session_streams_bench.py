"""Sessions whose streams have their own timelines (af_session_push_streams) on the cfg5 shape: 1024 streams of 48 kHz mono
f32, 80 mels, VAD on, device rows.  Five legs, alternated tick by tick in one process:
  lockstep         af_session_push of 960 samples, exactly as bench.py's measure_cfg5 does it;
  equal_streams    af_session_push_streams with every count 960 (the lockstep tick, selected from the counts);
  ragged           seeded counts in 960 +- 480 (mean 960), about 1 % of the streams ending (and restarting) per tick;
  ragged_441       the same at 44.1 kHz, 882 +- 441: every stream's resampling fractions are computed and uploaded;
  rings_available  the host loop: af_session_push_rings_available(max 1440) from pinned capture rings filled raggedly,
                   gated wire output (PCM16 + base64) to pinned host rows, then af_session_wire.
Per leg: p50 / p99 / mean host time per tick (every push ends in a stream synchronise), kernels launched per tick
(af_kernel_launch_count), bytes copied host-to-device and device-to-host per tick (computed from the tick's shapes), and
the device name and power limit read through NVML in the same run.  Prints one JSON line.

    timeout 900 python tools/session_streams_bench.py [--ticks 500]
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

TICK_DESC_BYTES = 64 + 4          # per stream and ragged tick: sizeof(StreamTick) + its uint32 frame count


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=500, help="timed ticks per leg (after 20 untimed ones)")
    ap.add_argument("--streams", type=int, default=1024)
    args = ap.parse_args()
    import torch
    import audioflow as af
    from audioflow import synth

    S, warm = args.streams, 20
    af.init(0)
    L = af.load_library()
    dev = torch.device("cuda:0")
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=True))
    x48 = synth.torch_batch(S, 4.0, 48000, 1, dev, seed=0)
    x441 = synth.torch_batch(S, 4.0, 44100, 1, dev, seed=1)
    x_host = x48[:, :48000].cpu().numpy()
    pcm = torch.empty((S, 1024), device=dev)
    lm = torch.empty((S, 16 * 80), device=dev)
    vad = torch.zeros((S, 16), device=dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 1024, lm.data_ptr(), 16 * 80, vad.data_ptr(), 16, None, 0, None)
    u32p, u8p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)

    def session(rate, max_tick, wire_mem=None):
        h = C.c_void_p()
        af._check(L.af_session_create(pipe._h, S, rate, 1, af.AF_FMT_F32, max_tick, C.byref(h)))
        if wire_mem is not None:
            af._check(L.af_session_enable_wire(h, C.byref(af.WireConfigC(1, 1, 1, wire_mem))))
        return h

    legs = {"lockstep": session(48000, 960), "equal_streams": session(48000, 960), "ragged": session(48000, 1440),
            "ragged_441": session(44100, 1323), "rings_available": session(48000, 1440, af.AF_MEM_HOST)}
    rng = np.random.default_rng(0)
    rings = [af.RingBuffer(16 * 1440) for _ in range(S)]
    ring_arr = (C.c_void_p * S)(*[r._h for r in rings])
    wticks = (af.WireTickC * S)()
    pp, ps, bp, bs, ff = C.c_void_p(), C.c_uint64(), C.c_void_p(), C.c_uint64(), C.c_uint64()
    npcm, nv = np.zeros(S, np.uint32), np.zeros(S, np.uint32)
    equal = np.full(S, 960, np.uint32)
    pos = {"ragged": 0, "ragged_441": 0}
    fed = np.zeros(S, np.int64)
    lat = {k: [] for k in legs}
    launches, h2d, d2h = ({k: 0 for k in legs} for _ in range(3))
    names = list(legs)
    torch.cuda.synchronize()
    for t in range(warm + args.ticks):
        off = (t % 100) * 960
        # this tick's ragged plans and the capture callbacks' ring writes: not timed
        plans = {}
        for leg, (mean, x) in (("ragged", (960, x48)), ("ragged_441", (882, x441))):
            n = rng.integers(mean // 2, mean + mean // 2 + 1, S).astype(np.uint32)
            end = (rng.random(S) < 0.01).astype(np.uint8)
            if pos[leg] + 1440 > x.shape[1]:
                pos[leg] = 0
            plans[leg] = (n, end, x.data_ptr() + pos[leg] * 4, x.shape[1])
            pos[leg] += mean
        for i in range(S):
            n = int(rng.integers(480, 1441))
            if fed[i] + n > x_host.shape[1]:
                fed[i] = 0
            rings[i].write(x_host[i, fed[i]:fed[i] + n])
            fed[i] += n
        ring_avail = np.array([min(1440, r.available()) for r in rings], np.int64) if t >= warm else None
        ring_end = (rng.random(S) < 0.01).astype(np.uint8)
        order = names[t % len(names):] + names[:t % len(names)]      # alternate which leg goes first
        for leg in order:
            h = legs[leg]
            l0 = L.af_kernel_launch_count()
            t0 = time.perf_counter()
            if leg == "lockstep":
                af._check(L.af_session_push(h, x48.data_ptr() + off * 4, x48.shape[1], 960, af.AF_MEM_DEVICE, C.byref(o),
                                            None, None, None))
            elif leg == "equal_streams":
                af._check(L.af_session_push_streams(h, x48.data_ptr() + off * 4, x48.shape[1], equal.ctypes.data_as(u32p), None,
                                                    af.AF_MEM_DEVICE, C.byref(o), None, None, None))
            elif leg == "rings_available":
                af._check(L.af_session_push_rings_available(h, ring_arr, 1440, ring_end.ctypes.data_as(u8p), None,
                                                            npcm.ctypes.data_as(u32p), None, nv.ctypes.data_as(u32p)))
                af._check(L.af_session_wire(h, C.byref(pp), C.byref(ps), C.byref(bp), C.byref(bs), wticks, C.byref(ff)))
            else:
                n, end, ptr, stride = plans[leg]
                af._check(L.af_session_push_streams(h, ptr, stride, n.ctypes.data_as(u32p), end.ctypes.data_as(u8p),
                                                    af.AF_MEM_DEVICE, C.byref(o), npcm.ctypes.data_as(u32p), None, None))
            dt = time.perf_counter() - t0
            if t < warm:
                continue
            lat[leg].append(dt)
            launches[leg] += L.af_kernel_launch_count() - l0
            if leg in ("ragged", "ragged_441"):
                h2d[leg] += S * TICK_DESC_BYTES + (4 * int(npcm.sum()) if leg == "ragged_441" else 0)   # plan + fractions
            elif leg == "rings_available":
                mx = int(ring_avail.max())
                h2d[leg] += S * TICK_DESC_BYTES + 4 * ((S - 1) * mx + int(ring_avail[-1]))   # plan + input rows
                n = int(nv.max()) * 160                                  # gated payload bound: the most frames x hop
                d2h[leg] += S * (C.sizeof(af.WireTickC) + 2 * n + (L.af_pcm16_base64_len(n) if n else 0))
    for h in legs.values():
        L.af_session_destroy(h)
    res = {"tool": "session_streams_bench", "streams": S, "n_mels": 80, "vad": True, "ticks": args.ticks, "warmup_ticks": warm,
           "end_fraction_per_tick": 0.01}
    for leg, v in lat.items():
        a = np.array(v) * 1e3
        res[leg] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "mean_ms": float(a.mean()),
                    "kernel_launches_per_tick": launches[leg] / args.ticks, "h2d_bytes_per_tick": h2d[leg] / args.ticks,
                    "d2h_bytes_per_tick": d2h[leg] / args.ticks}
    res.update(device_info(0))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
