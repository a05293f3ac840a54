"""Sessions of mixed capture formats (af_session_create_formats) on the cfg5 shape: 1024 streams, 80 mels, VAD on, wire
off, device rows.  The mix is 512 x 48 kHz mono, 256 x 44.1 kHz mono, 128 x 48 kHz stereo and 128 x 16 kHz mono, f32.
Three legs, alternated tick by tick in one process:
  mixed          one mixed session, every stream pushing its own 20 ms (960, 882, 1920, 320 samples);
  four_sessions  the same streams as four single-format sessions, pushed one after another (lockstep ticks); a tick is
                 the time of all four;
  mixed_ragged   the mixed session with counts of 20 ms +- 50 % in whole frames, about 1 % of the streams ending per tick
                 and restarting in another format before the next tick.
Per leg: p50 / p99 / mean host time per tick (every push ends in a stream synchronise), kernels launched per tick
(af_kernel_launch_count), bytes uploaded per tick (counted from the shapes: the per-stream tick plan and the 44.1 kHz
fraction slices, one per distinct plan), and the device name and power limit read through NVML in the same run.  Prints
one JSON line.

    timeout 900 python tools/session_formats_bench.py [--ticks 500]
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

TICK_DESC_BYTES = 64 + 4          # per stream and per-stream tick: sizeof(StreamTick) + its uint32 frame count
# (rate, channels, 20 ms of samples, streams)
MIX = [(48000, 1, 960, 512), (44100, 1, 882, 256), (48000, 2, 1920, 128), (16000, 1, 320, 128)]
TABLE = 1                         # the format resampled through a fraction table (44.1 kHz)
N441 = 320                        # 16 kHz samples of 882 samples at 44.1 kHz (a slice of fractions per distinct plan)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=500, help="timed ticks per leg (after 20 untimed ones)")
    args = ap.parse_args()
    import torch
    import audioflow as af
    from audioflow import synth

    warm = 20
    af.init(0)
    L = af.load_library()
    dev = torch.device("cuda:0")
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=True))
    sf = np.concatenate([np.full(n, i, np.uint32) for i, (_, _, _, n) in enumerate(MIX)])
    S = sf.size
    row0 = np.concatenate([[0], np.cumsum([m[3] for m in MIX])])
    bound = np.array([MIX[f][2] for f in sf], np.int64)
    x = synth.torch_batch(S, 4.0, 48000, 2, dev, seed=0)                    # every row read as its stream's format
    W = x.shape[1]
    pcm = torch.empty((S, 1024), device=dev)
    lm = torch.empty((S, 16 * 80), device=dev)
    vad = torch.zeros((S, 16), device=dev, dtype=torch.uint8)

    def outputs(r0):
        return af.OutputsC(pcm.data_ptr() + r0 * 1024 * 4, 1024, lm.data_ptr() + r0 * 16 * 80 * 4, 16 * 80,
                           vad.data_ptr() + r0 * 16, 16, None, 0, None)

    o = outputs(0)
    u32p, u8p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)
    fmts = (af.StreamFormatC * len(MIX))(*[af.StreamFormatC(r, c, 0, n * 3 // 2) for r, c, n, _ in MIX])

    def mixed():
        h = C.c_void_p()
        af._check(L.af_session_create_formats(pipe._h, S, fmts, len(MIX), sf.ctypes.data_as(u32p), af.AF_FMT_F32, C.byref(h)))
        return h

    mixed_h, ragged_h = mixed(), mixed()
    singles = []
    for i, (r, c, n, cnt) in enumerate(MIX):
        h = C.c_void_p()
        af._check(L.af_session_create(pipe._h, cnt, r, c, af.AF_FMT_F32, n * 3 // 2, C.byref(h)))
        singles.append((h, int(row0[i]), n, outputs(int(row0[i]))))
    own = bound.astype(np.uint32)
    npcm = np.zeros(S, np.uint32)
    rng = np.random.default_rng(0)
    cur_fmt = sf.copy()                                                      # mixed_ragged: every stream's format
    life = np.zeros(S, np.int64)                                             # frames pushed in the current life
    last = np.zeros(S, np.int64)                                             # the last tick's frames
    fresh = np.ones(S, bool)
    names = ["mixed", "four_sessions", "mixed_ragged"]
    lat = {k: [] for k in names}
    launches, h2d = ({k: 0 for k in names} for _ in range(2))
    torch.cuda.synchronize()
    for t in range(warm + args.ticks):
        off = (t % 100) * 1920
        ptr = x.data_ptr() + off * 4
        # this tick's ragged counts and ends: not timed
        c_r = np.array([MIX[f][1] for f in cur_fmt], np.int64)
        b_r = np.array([MIX[f][2] for f in cur_fmt], np.int64) // c_r
        n_r = (rng.integers(b_r // 2, b_r + b_r // 2 + 1) * c_r).astype(np.uint32)
        end = (rng.random(S) < 0.01).astype(np.uint8)
        order = names[t % len(names):] + names[:t % len(names)]              # alternate which leg goes first
        for leg in order:
            l0 = L.af_kernel_launch_count()
            t0 = time.perf_counter()
            if leg == "mixed":
                af._check(L.af_session_push_streams(mixed_h, ptr, W, own.ctypes.data_as(u32p), None, af.AF_MEM_DEVICE,
                                                    C.byref(o), npcm.ctypes.data_as(u32p), None, None))
            elif leg == "four_sessions":
                for h, r0, n, og in singles:
                    af._check(L.af_session_push(h, ptr + r0 * W * 4, W, n, af.AF_MEM_DEVICE, C.byref(og), None, None, None))
            else:
                af._check(L.af_session_push_streams(ragged_h, ptr, W, n_r.ctypes.data_as(u32p), end.ctypes.data_as(u8p),
                                                    af.AF_MEM_DEVICE, C.byref(o), npcm.ctypes.data_as(u32p), None, None))
            dt = time.perf_counter() - t0
            if leg == "mixed_ragged":
                # bytes: one fraction slice per distinct 44.1 kHz plan (a plan is a function of the format, the frames
                # of the life so far, the last tick's frames, this tick's count and the end flag)
                frames = n_r.astype(np.int64) // c_r
                keys = {}
                for k in np.nonzero(cur_fmt == TABLE)[0]:
                    key = (bool(fresh[k]), 0 if fresh[k] else int(life[k]), 0 if fresh[k] else int(last[k]), int(n_r[k]),
                           int(end[k]))
                    keys.setdefault(key, int(npcm[k]))
                frac_bytes = 4 * sum(keys.values())
                life = np.where(fresh, frames, life + frames)
                last, fresh = frames, end.astype(bool)
                ended = np.nonzero(end)[0]
                new = ((cur_fmt[ended] + 1 + rng.integers(0, 3, ended.size)) % len(MIX)).astype(np.uint32)
                af._check(L.af_session_restart_streams(ragged_h, ended.astype(np.uint32).ctypes.data_as(u32p),
                                                       new.ctypes.data_as(u32p), ended.size))
                cur_fmt[ended] = new
            if t < warm:
                continue
            lat[leg].append(dt)
            launches[leg] += L.af_kernel_launch_count() - l0
            if leg == "mixed":                    # the plan; the 44.1 kHz streams share one plan and one slice
                h2d[leg] += S * TICK_DESC_BYTES + 4 * N441
            elif leg == "four_sessions":          # lockstep: the plan goes in kernel parameters; one 44.1 kHz slice
                h2d[leg] += 4 * N441
            else:
                h2d[leg] += S * TICK_DESC_BYTES + frac_bytes
    for h in [mixed_h, ragged_h] + [s[0] for s in singles]:
        L.af_session_destroy(h)
    res = {"tool": "session_formats_bench", "streams": S, "mix": [list(m) for m in MIX], "n_mels": 80, "vad": True,
           "wire": False, "ticks": args.ticks, "warmup_ticks": warm, "end_fraction_per_tick": 0.01}
    for leg, v in lat.items():
        a = np.array(v) * 1e3
        res[leg] = {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "mean_ms": float(a.mean()),
                    "kernel_launches_per_tick": launches[leg] / args.ticks, "h2d_bytes_per_tick": h2d[leg] / args.ticks}
    res.update(device_info(0))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
