"""Wire segment table (af_session_enable_wire_segments) on the cfg5 shape: 1024 streams x 960-sample 48 kHz mono f32
ticks, 80 mels, VAD on, gated wire output as PCM16 and base64 in device rows, with pre-roll 0 and 30 frames.
Per pre-roll, sessions that differ only in the table -- off, on with device rows, on with pinned host rows -- are pushed
alternately tick by tick from the same device input (the leg that goes first rotates); 500 timed ticks after 20 untimed
ones.  Per leg: p50 / p90 / mean host time per tick (every push ends in a stream synchronise), kernels launched per tick
(af_kernel_launch_count) and the pieces per tick; plus the device name and power limit read through NVML in the same
run.  Prints one JSON line.

--tree DIR imports the package (and so the library) of another checkout, e.g. the parent commit built beside this one;
a library without the table runs the "off" leg alone, so the same script times the parent and this change.

    timeout 900 python tools/session_wire_segments_bench.py [--ticks 500] [--tree DIR]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=500, help="timed ticks per leg (after 20 untimed ones)")
    ap.add_argument("--streams", type=int, default=1024)
    ap.add_argument("--tree", default=ROOT, help="checkout whose audioflow package and library to time")
    args = ap.parse_args()
    tree = os.path.abspath(args.tree)
    for p in (os.path.join(ROOT, "tools"), os.path.join(tree, "audio-flow-rs_b200")):
        sys.path.insert(0, p)
    import numpy as np
    import torch
    import audioflow as af
    from audioflow import synth
    from session_wire_bench import device_info

    S, tick, warm, M = args.streams, 960, 20, 80
    af.init(0)
    L = af.load_library()
    has_table = hasattr(L, "af_session_enable_wire_segments")
    dev = torch.device("cuda:0")
    pipe = af.Pipeline(af.pipeline_config(n_mels=M, vad_enable=True))
    x = synth.torch_batch(S, 2.0, 48000, 1, dev, seed=0)
    pcm = torch.empty((S, 512), device=dev)
    lm = torch.empty((S, 8 * M), device=dev)
    vad = torch.zeros((S, 16), device=dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 512, lm.data_ptr(), 8 * M, vad.data_ptr(), 16, None, 0, None)
    nf = np.zeros(S, np.uint32)
    nseg = np.zeros(S, np.uint32)
    u32p = C.POINTER(C.c_uint32)
    rows, stride = C.c_void_p(), C.c_uint64()
    wt = (af.WireTickC * S)()

    def session(table, preroll):
        h = C.c_void_p()
        af._check(L.af_session_create(pipe._h, S, 48000, 1, af.AF_FMT_F32, tick, C.byref(h)))
        cfg = af.WireConfigC(1, 1, 1, af.AF_MEM_DEVICE)
        af._check(L.af_session_enable_wire(h, C.byref(cfg)))
        af._check(L.af_session_set_wire_preroll(h, preroll))
        if table is not None:
            af._check(L.af_session_enable_wire_segments(h, 1, table))
        return h

    res = {"tool": "session_wire_segments_bench", "tree": "this" if tree == ROOT else os.path.basename(tree),
           "table_in_library": has_table, "streams": S, "tick_samples": tick, "rate": 48000, "n_mels": M, "vad": True,
           "gate": 1, "pcm16": 1, "base64": 1, "wire_mem": "device", "ticks": args.ticks, "warmup_ticks": warm}
    for P in (0, 30):
        legs = {"off": session(None, P)}
        if has_table:
            legs["on_device_rows"] = session(af.AF_MEM_DEVICE, P)
            legs["on_host_rows"] = session(af.AF_MEM_HOST, P)
        names = list(legs)
        lat = {k: [] for k in legs}
        launches = {k: 0 for k in legs}
        pieces = {k: 0 for k in legs}
        torch.cuda.synchronize()
        for t in range(warm + args.ticks):
            off = (t % 100) * tick
            r = t % len(names)
            for leg in names[r:] + names[:r]:
                h = legs[leg]
                l0 = L.af_kernel_launch_count()
                t0 = time.perf_counter()
                af._check(L.af_session_push(h, x.data_ptr() + off * 4, x.shape[1], tick, af.AF_MEM_DEVICE, C.byref(o),
                                            None, nf.ctypes.data_as(u32p), None))
                af._check(L.af_session_wire(h, None, None, None, None, wt, None))
                if leg != "off":
                    af._check(L.af_session_wire_segments(h, C.byref(rows), C.byref(stride), nseg.ctypes.data_as(u32p)))
                dt = time.perf_counter() - t0
                if t < warm:
                    continue
                lat[leg].append(dt)
                launches[leg] += L.af_kernel_launch_count() - l0
                if leg != "off":
                    pieces[leg] += int(nseg.sum())
        for h in legs.values():
            L.af_session_destroy(h)
        out = {}
        for leg, v in lat.items():
            a = np.array(v) * 1e6
            out[leg] = {"p50_us": float(np.percentile(a, 50)), "p90_us": float(np.percentile(a, 90)), "mean_us": float(a.mean()),
                        "kernel_launches_per_tick": launches[leg] / args.ticks, "pieces_per_tick": pieces[leg] / args.ticks}
        res[f"preroll_{P}"] = out
    res.update(device_info(0))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
