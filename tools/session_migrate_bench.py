"""Stream records: what moving live streams between sessions costs, on the cfg5 shape (1024 x 20 ms at 48 kHz mono, 80
mels, VAD on, device rows, wire off).

Legs alternated tick by tick, each on its own sessions:
  plain        the lockstep tick of a session that never moves a stream (the reference leg);
  move_host    a tick of session A, then 1 % of its streams (10) exported to host records, imported into free slots of
               session B and reset in A (A ticks per stream from the first move on: its reset slots restart);
  move_device  the same through device records on the same GPU;
  move_peer    (two GPUs) move_host with B on GPU 1.
Per leg: p50 / p99 / mean host time of the tick plus the move (every call ends in a stream synchronise), and of the move
alone.  Then one whole-session move, repeated: 1024 streams exported and imported into a 2048-slot session (host and
device records), and the imported session's next ticks -- the per-stream tick, since its other 1024 slots stand elsewhere
-- beside the lockstep tick.  The device name and power limit are read through NVML in the same run.  Prints one JSON line.

    timeout 900 python tools/session_migrate_bench.py [--ticks 500]
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

S, TICK, MOVE = 1024, 960, 10


def _stats(a):
    a = np.asarray(a) * 1e6
    return {"p50_us": float(np.percentile(a, 50)), "p99_us": float(np.percentile(a, 99)), "mean_us": float(a.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=500, help="timed ticks per leg (after 20 untimed ones)")
    ap.add_argument("--whole", type=int, default=20, help="timed whole-session moves per record kind")
    args = ap.parse_args()
    import torch
    import audioflow as af
    from audioflow import synth
    af.init(0)
    L = af.load_library()
    u32p = C.POINTER(C.c_uint32)
    n_gpus = C.c_int(0)
    L.af_device_count(C.byref(n_gpus))
    dev = torch.device("cuda:0")
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=True))
    # input and output rows for the largest session (2 S streams): a tick reads and writes one row per stream
    x = synth.torch_batch(2 * S, 4.0, 48000, 1, dev, seed=3)
    W = x.shape[1]
    pcm = torch.empty((2 * S, 512), device=dev)
    lm = torch.empty((2 * S, 8 * 80), device=dev)
    vad = torch.zeros((2 * S, 16), device=dev, dtype=torch.uint8)
    o = af.OutputsC(pcm.data_ptr(), 512, lm.data_ptr(), 8 * 80, vad.data_ptr(), 16, None, 0, None)

    def session(n, device=0):
        af.init(device)
        s = af.Session(pipe, n, 48000, 1, af.AF_FMT_F32, max_tick_samples=TICK)
        af.init(0)
        return s

    def push(s, t):
        assert s.S <= x.shape[0] and s.S <= pcm.shape[0]
        af._check(L.af_session_push(s._h, x.data_ptr() + (t % 150) * TICK * 4, W, TICK, af.AF_MEM_DEVICE, C.byref(o),
                                    None, None, None))

    legs = ["plain", "move_host", "move_device"] + (["move_peer"] if n_gpus.value >= 2 else [])
    src = {k: session(S) for k in legs}
    dst = {k: session(S, 1 if k == "move_peer" else 0) for k in legs if k != "plain"}
    rb = src["plain"].record_bytes()
    host_rec = np.zeros((MOVE, rb), np.uint8)
    dev_rec = torch.zeros((MOVE, rb), dtype=torch.uint8, device=dev)
    rng = np.random.default_rng(0)
    lat = {k: [] for k in legs}
    move = {k: [] for k in legs if k != "plain"}
    warm = 20
    next_slot = {k: 0 for k in dst}
    torch.cuda.synchronize()
    for t in range(warm + args.ticks):
        ids = np.ascontiguousarray(rng.choice(S, MOVE, replace=False), np.uint32)
        order = legs[t % len(legs):] + legs[:t % len(legs)]
        for leg in order:
            s = src[leg]
            t0 = time.perf_counter()
            push(s, t)
            t1 = time.perf_counter()
            if leg != "plain":
                d = dst[leg]
                slots = np.ascontiguousarray((next_slot[leg] + np.arange(MOVE)) % S, np.uint32)
                next_slot[leg] = (next_slot[leg] + MOVE) % S
                ptr, mem = (dev_rec.data_ptr(), af.AF_MEM_DEVICE) if leg == "move_device" else (host_rec.ctypes.data, af.AF_MEM_HOST)
                af._check(L.af_session_export_streams(s._h, ids.ctypes.data_as(u32p), MOVE, ptr, mem))
                af._check(L.af_session_import_streams(d._h, slots.ctypes.data_as(u32p), ptr, MOVE, None, mem))
                af._check(L.af_session_reset_streams(s._h, ids.ctypes.data_as(u32p), MOVE))
            t2 = time.perf_counter()
            if t >= warm:
                lat[leg].append(t2 - t0)
                if leg != "plain":
                    move[leg].append(t2 - t1)
    out = {"tool": "session_migrate_bench", "shape": "cfg5", "streams": S, "tick_samples": TICK, "ticks": args.ticks,
           "warmup_ticks": warm, "moved_per_tick": MOVE, "record_bytes": rb, "gpus": n_gpus.value}
    for leg in legs:
        out[leg] = {"tick_plus_move": _stats(lat[leg])}
        if leg != "plain":
            out[leg]["move_only"] = _stats(move[leg])

    # one whole-session move: 1024 streams into a 2048-slot session, then that session's ticks beside the lockstep one
    a, big = session(S), session(2 * S)
    for t in range(8):
        push(a, t)
    ids = np.arange(S, dtype=np.uint32)
    slots = np.ascontiguousarray(np.random.default_rng(1).permutation(2 * S)[:S], np.uint32)
    whole_host = np.zeros((S, rb), np.uint8)
    whole_dev = torch.zeros((S, rb), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    whole = {"host": [], "device": []}
    for r in range(args.whole + 2):
        for kind, (ptr, mem) in (("host", (whole_host.ctypes.data, af.AF_MEM_HOST)),
                                 ("device", (whole_dev.data_ptr(), af.AF_MEM_DEVICE))):
            t0 = time.perf_counter()
            af._check(L.af_session_export_streams(a._h, ids.ctypes.data_as(u32p), S, ptr, mem))
            af._check(L.af_session_import_streams(big._h, slots.ctypes.data_as(u32p), ptr, S, None, mem))
            if r >= 2:
                whole[kind].append(time.perf_counter() - t0)
    out["whole_session_move"] = {k: _stats(v) for k, v in whole.items()}
    out["whole_session_move"]["records"] = S
    tick_ps, tick_ls = [], []
    big2 = session(2 * S)
    for t in range(8, 8 + 200):
        for s, acc in ((big, tick_ps), (big2, tick_ls)):
            t0 = time.perf_counter()
            push(s, t)
            acc.append(time.perf_counter() - t0)
    out["after_whole_move_2048"] = {"per_stream_tick": _stats(tick_ps[20:]), "lockstep_tick_same_size": _stats(tick_ls[20:])}
    out.update(device_info(0))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
