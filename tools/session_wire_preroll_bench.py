"""Wire pre-roll (af_session_set_wire_preroll) on the cfg5 shape: 1024 streams x 960-sample 48 kHz mono f32 ticks,
80 mels, VAD on, gated wire output as PCM16 and base64 with its features.  Two runs: the wire rows and the feature rows on
the device, then both in pinned host rows.  In each run two sessions, one with pre-roll 0 and one with pre-roll P (30
frames, 300 ms), are pushed alternately tick by tick from the same device input (the leg that goes first alternates too);
500 timed ticks after 20 untimed ones.
Per leg: p50 / p99 / mean host time per tick (every push ends in a stream synchronise), kernels launched per tick
(af_kernel_launch_count), bytes copied device-to-host per tick and the bytes of the payload rows themselves, both computed
from the tick's counts; plus the device name and power limit read through NVML in the same run.  Prints one JSON line.

    timeout 900 python tools/session_wire_preroll_bench.py [--ticks 500] [--preroll 30]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=500, help="timed ticks per leg (after 20 untimed ones)")
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--preroll", type=int, default=30, help="frames of pre-roll of the second leg")
    args = ap.parse_args()
    import torch
    import audioflow as af
    from audioflow import synth

    S, tick, warm, M = args.streams, 960, 20, 80
    af.init(0)
    L = af.load_library()
    dev = torch.device("cuda:0")
    pipe = af.Pipeline(af.pipeline_config(n_mels=M, vad_enable=True))
    x = synth.torch_batch(S, 2.0, 48000, 1, dev, seed=0)
    pcm = torch.empty((S, 512), device=dev)
    lm = torch.empty((S, 8 * M), device=dev)
    vad = torch.zeros((S, 16), device=dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 512, lm.data_ptr(), 8 * M, vad.data_ptr(), 16, None, 0, None)
    nf = np.zeros(S, np.uint32)
    kept = np.zeros(S, np.uint32)
    u32p = C.POINTER(C.c_uint32)
    rows, stride = C.c_void_p(), C.c_uint64()
    tick_rec = C.sizeof(af.WireTickC)

    P = args.preroll
    wt = (af.WireTickC * S)()

    def session(mem, preroll):
        h = C.c_void_p()
        af._check(L.af_session_create(pipe._h, S, 48000, 1, af.AF_FMT_F32, tick, C.byref(h)))
        cfg = af.WireConfigC(1, 1, 1, mem)
        af._check(L.af_session_enable_wire(h, C.byref(cfg)))
        af._check(L.af_session_enable_wire_features(h, 1, mem))
        af._check(L.af_session_set_wire_preroll(h, preroll))
        return h

    res = {"tool": "session_wire_preroll_bench", "streams": S, "tick_samples": tick, "rate": 48000, "n_mels": M, "vad": True,
           "gate": 1, "pcm16": 1, "base64": 1, "features": 1, "preroll_frames": P, "ticks": args.ticks, "warmup_ticks": warm}
    for run, mem in (("device_rows", af.AF_MEM_DEVICE), ("host_rows", af.AF_MEM_HOST)):
        legs = {"preroll_0": session(mem, 0), f"preroll_{P}": session(mem, P)}
        names = list(legs)
        lat = {k: [] for k in legs}
        launches = {k: 0 for k in legs}
        d2h = {k: 0 for k in legs}
        payload = {k: 0 for k in legs}
        torch.cuda.synchronize()
        for t in range(warm + args.ticks):
            off = (t % 100) * tick
            for leg in (names if t % 2 == 0 else names[::-1]):
                h = legs[leg]
                l0 = L.af_kernel_launch_count()
                t0 = time.perf_counter()
                af._check(L.af_session_push(h, x.data_ptr() + off * 4, x.shape[1], tick, af.AF_MEM_DEVICE, C.byref(o),
                                            None, nf.ctypes.data_as(u32p), None))
                af._check(L.af_session_wire_features(h, C.byref(rows), C.byref(stride), kept.ctypes.data_as(u32p)))
                af._check(L.af_session_wire(h, None, None, None, None, wt, None))
                dt = time.perf_counter() - t0
                if t < warm:
                    continue
                lat[leg].append(dt)
                launches[leg] += L.af_kernel_launch_count() - l0
                T = int(nf.max())                                  # the tick's frames, and the pre-roll bound every payload
                F = T + (P if T and leg != "preroll_0" else 0)
                n = F * 160
                b = S * tick_rec + S * 4                           # the wire's tick records, the feature counts
                if mem == af.AF_MEM_HOST:                          # gated PCM16 + base64 rows and feature rows, bounded
                    b += S * (2 * n + (L.af_pcm16_base64_len(n) if n else 0)) + S * F * M * 4
                d2h[leg] += b
                ns = sum(int(r.n_samples) for r in wt)
                payload[leg] += 2 * ns + sum(int(r.n_chars) for r in wt) + int(kept.sum()) * M * 4
        for h in legs.values():
            L.af_session_destroy(h)
        out = {}
        for leg, v in lat.items():
            a = np.array(v) * 1e6
            out[leg] = {"p50_us": float(np.percentile(a, 50)), "p99_us": float(np.percentile(a, 99)), "mean_us": float(a.mean()),
                        "kernel_launches_per_tick": launches[leg] / args.ticks, "d2h_bytes_per_tick": d2h[leg] / args.ticks,
                        "payload_bytes_per_tick": payload[leg] / args.ticks}
        res[run] = out
    res.update(device_info(0))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
