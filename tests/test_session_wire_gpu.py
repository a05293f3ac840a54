"""The streaming wire output of sessions (af_session_enable_wire / af_session_wire): per tick and stream, the PCM16 samples
and the base64 text WebSocketClient::send_audio sends (websocket.rs:244-254), ungated or gated to the speech segments
(specs/0001-spec.md:466), with the segment events of the tick.  Everything is bit-exact against the oracle objects fed the
same chunks: BatchResampler::process per tick, the framed VAD over the concatenated PCM, orc_vad_segments / orc_vad_gate
over the whole session."""
import base64
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPEECH, ENDING = 1, 2


def _ref_pcm(orc, x, rate, ch, fmt, tick, n_ticks):
    """Per-tick BatchResampler::process outputs of one stream (no flush)."""
    xi = orc.i16_to_f32(x) if fmt == "i16" else x
    mono = orc.to_mono(xi, ch)
    b = orc.BatchResampler(rate, 16000)
    return [b.process(mono[t * tick:(t + 1) * tick]) for t in range(n_ticks)]


def _b64(pcm16):
    return base64.b64encode(np.asarray(pcm16, np.int16).astype("<i2").tobytes())


def _bursts(seed, seconds, rate):
    """Short tone bursts between quiet stretches: segments open and close many times per 200 ms."""
    rng = np.random.default_rng(seed)
    n = int(seconds * rate)
    x = rng.normal(0.0, 1e-3, n)
    pos, loud = 0, bool(seed & 1)
    while pos < n:
        m = int(rng.uniform(0.02, 0.09) * rate)
        if loud:
            t = np.arange(min(m, n - pos)) / rate
            x[pos:pos + m] += 0.1 * np.sin(2 * np.pi * rng.uniform(200, 3000) * t)
        pos += m
        loud = not loud
    return np.clip(x, -1, 1).astype(np.float32)


def _oracle_events(orc, states, frames_per_tick, hop):
    """Per tick: (first_frame, started, ended, in_speech, continued, kept samples) binned from orc_vad_segments."""
    segs = orc.vad_segments(states)
    T = len(states)
    close = []
    for s, e in segs:
        if e < T:
            close.append(e - 1 if states[e - 1] == ENDING else e)          # Ending closes inclusive, Silence exclusive
        elif states[T - 1] == ENDING:
            close.append(T - 1)
    close = np.array(close, np.int64)
    kept = np.zeros(T, bool)
    for s, e in segs:
        kept[s:e] = True
    out, F = [], 0
    for n in frames_per_tick:
        lo, hi = F, F + n
        started = int(((segs[:, 0] >= lo) & (segs[:, 0] < hi)).sum()) if len(segs) else 0
        ended = int(((close >= lo) & (close < hi)).sum())
        last = hi - 1
        in_speech = last >= 0 and states[last] == SPEECH
        cont = 0
        if lo > 0 and states[lo - 1] == SPEECH:
            for s, e in segs:
                if s <= lo - 1 < e:
                    cont = (min(e, hi) - lo) * hop
        out.append((lo, started, ended, bool(in_speech), cont, int(kept[lo:hi].sum()) * hop))
        F = hi
    return out, segs


def _device_rows(ptr, rows, stride, dtype):
    """Copy [rows, stride] elements of a device buffer to the host (through torch's __cuda_array_interface__ support)."""
    import torch

    class _Rows:
        @property
        def __cuda_array_interface__(self):
            return {"shape": (rows, stride), "typestr": np.dtype(dtype).str, "data": (ptr, False), "version": 2, "strides": None}
    return torch.as_tensor(_Rows(), device="cuda").cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rate,tick,fmt,ch", [(48000, 960, "f32", 1), (44100, 882, "f32", 1), (48000, 1000, "i16", 2),
                                               (16000, 320, "f32", 1), (32000, 77, "f32", 1)])
def test_wire_ungated_matches_oracle(af, orc, rate, tick, fmt, ch):
    from audioflow import synth
    S, n_ticks = 3, 40
    total = tick * n_ticks
    xs = [synth.stream(60 + i, total / rate + 0.01, rate, ch, fmt)[: total * ch] for i in range(S)]
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=80)), S, rate, ch, af.AF_FMT_I16 if fmt == "i16" else af.AF_FMT_F32,
                     max_tick_samples=tick * ch)
    ses.enable_wire(gate=False)
    refs = [_ref_pcm(orc, xs[i], rate, ch, fmt, tick, n_ticks) for i in range(S)]
    frames = 0
    for t in range(n_ticks):
        r = ses.push(np.stack([x[t * tick * ch:(t + 1) * tick * ch] for x in xs]))
        w = ses.wire()
        assert w["first_frame"] == frames
        frames += r["n_frames"]
        for i in range(S):
            got, ref = w["streams"][i], refs[i][t]
            want = orc.pcm16_encode(ref)
            assert got["n_samples"] == len(ref) and got["continued"] == 0
            assert np.array_equal(got["pcm16"], want), (t, i)
            assert got["base64"] == orc.pcm16_base64(ref) == _b64(want), (t, i)
            assert got["n_chars"] == len(got["base64"]) == af.load_library().af_pcm16_base64_len(len(ref))


FRAMINGS = {"stft": dict(n_mels=80), "20ms": dict(n_mels=0, vad_frame_len=320, vad_hop=320)}


def _gated_run(af, orc, framing, tick, n_ticks, vad_cfg, mem=None, rings=False, reps=1):
    """Streams 0-1: tone bursts, 2-3: the synthetic speech-like signal.  Returns (xs, per-pass list of per-tick wire())."""
    from audioflow import synth
    S, rate = 4, 48000
    secs = tick * n_ticks / rate + 0.01
    xs = [_bursts(7 + i, secs, rate)[: tick * n_ticks] for i in range(2)] + \
         [synth.stream(300 + i, secs, rate, 1)[: tick * n_ticks] for i in range(2)]
    pipe = af.Pipeline(af.pipeline_config(vad=af.VadConfig(**vad_cfg), **FRAMINGS[framing]))
    ses = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    ses.enable_wire(gate=True, mem=af.AF_MEM_HOST if mem is None else mem)
    passes = []
    for _ in range(reps):
        ticks = []
        ring = [af.RingBuffer(4 * tick) for _ in range(S)] if rings else None
        for t in range(n_ticks):
            chunk = [x[t * tick:(t + 1) * tick] for x in xs]
            if rings:
                for i in range(S):
                    assert ring[i].write(chunk[i]) == tick
                r = ses.push_rings(ring, tick)
            else:
                r = ses.push(np.stack(chunk))
            w = ses.wire()
            w["n_frames"] = r["n_frames"]
            if mem == af.AF_MEM_DEVICE:
                w["pcm16_rows"] = _device_rows(w["pcm16_ptr"], S, w["pcm16_stride"], np.int16)
                w["base64_rows"] = _device_rows(w["base64_ptr"], S, w["base64_stride"], np.uint8)
                for i, st in enumerate(w["streams"]):
                    st["pcm16"] = w["pcm16_rows"][i, :st["n_samples"]].copy()
                    st["base64"] = w["base64_rows"][i, :st["n_chars"]].tobytes()
            ticks.append(w)
        passes.append(ticks)
        ses.reset()
    return xs, passes


VAD_FAST = dict(threshold_db=-50.0, smoothing_factor=0.3, silence_timeout_frames=2, min_speech_frames=3)


@pytest.mark.gpu
@pytest.mark.parametrize("framing", ["stft", "20ms"])
@pytest.mark.parametrize("tick,vad_cfg", [(960, {}), (9600, VAD_FAST)])
def test_wire_gated_matches_oracle(af, orc, framing, tick, vad_cfg):
    n_ticks = 16 if tick == 9600 else 120
    frame_len, hop = (400, 160) if framing == "stft" else (320, 320)
    xs, (ticks,) = _gated_run(af, orc, framing, tick, n_ticks, vad_cfg)
    ovc = orc.default_vad_config()
    for k, v in vad_cfg.items():
        setattr(ovc, k, v)
    close_then_start = 0
    for i in range(len(xs)):
        ref_pcm = np.concatenate(_ref_pcm(orc, xs[i], 48000, 1, "f32", tick, n_ticks))
        states, _ = orc.VoiceActivityDetector(ovc).stream(ref_pcm, frame_len, hop)
        events, segs = _oracle_events(orc, states, [w["n_frames"] for w in ticks], hop)
        assert sum(w["n_frames"] for w in ticks) == len(states)
        want = orc.pcm16_encode(orc.vad_gate(ref_pcm, None, segs, hop)[0])
        got = np.concatenate([w["streams"][i]["pcm16"] for w in ticks])
        assert np.array_equal(got, want), f"stream {i}: gated payloads differ from orc_vad_gate"
        assert sum(w["streams"][i]["started"] for w in ticks) == len(segs)
        for t, (w, ev) in enumerate(zip(ticks, events)):
            g = w["streams"][i]
            assert (w["first_frame"], g["started"], g["ended"], g["in_speech"], g["continued"], g["n_samples"]) == ev, (i, t)
            assert g["base64"] == _b64(g["pcm16"]), (i, t)
            close_then_start += g["continued"] > 0 and g["started"] > 0
    if tick == 9600:
        assert close_then_start, "no tick finished an utterance and started a new one"


@pytest.mark.gpu
def test_wire_paths_agree(af, orc):
    """Host rows, device rows and ring-fed ticks give the same bytes."""
    _, (host,) = _gated_run(af, orc, "stft", 4800, 20, VAD_FAST)
    _, (dev,) = _gated_run(af, orc, "stft", 4800, 20, VAD_FAST, mem=af.AF_MEM_DEVICE)
    _, (ringed,) = _gated_run(af, orc, "stft", 4800, 20, VAD_FAST, rings=True)
    for a, b, c in zip(host, dev, ringed):
        assert a["first_frame"] == b["first_frame"] == c["first_frame"]
        for x, y, z in zip(a["streams"], b["streams"], c["streams"]):
            for k in ("started", "ended", "in_speech", "continued", "n_samples", "n_chars", "base64"):
                assert x[k] == y[k] == z[k], k
            assert np.array_equal(x["pcm16"], y["pcm16"]) and np.array_equal(x["pcm16"], z["pcm16"])


@pytest.mark.gpu
def test_wire_reset_replays(af, orc):
    _, (p0, p1) = _gated_run(af, orc, "20ms", 1920, 30, VAD_FAST, reps=2)
    for a, b in zip(p0, p1):
        assert a["first_frame"] == b["first_frame"]
        for x, y in zip(a["streams"], b["streams"]):
            for k in ("started", "ended", "in_speech", "continued", "n_samples", "base64"):
                assert x[k] == y[k], k
            assert np.array_equal(x["pcm16"], y["pcm16"])


@pytest.mark.gpu
def test_wire_special_values(af, orc):
    """A 16 kHz passthrough session hands the samples through unchanged: clamping, the +-Inf ends and NaN -> 0."""
    vals = np.array([0.5, -0.5, 1.0, -1.0, 3.0, -3.0, np.inf, -np.inf, np.nan, 0.0, 1e-6, -0.99999], np.float32)
    S, tick, n_ticks = 2, 320, 6
    rng = np.random.default_rng(11)
    xs = [rng.choice(vals, tick * n_ticks).astype(np.float32) for _ in range(S)]
    xs[0][:len(vals)] = vals
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False)), S, 16000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    ses.enable_wire(gate=False)
    for t in range(n_ticks):
        chunk = [x[t * tick:(t + 1) * tick] for x in xs]
        ses.push(np.stack(chunk))
        w = ses.wire()
        for i in range(S):
            g = w["streams"][i]
            assert np.array_equal(g["pcm16"], orc.pcm16_encode(chunk[i]))
            assert g["base64"] == orc.pcm16_base64(chunk[i]) == _b64(orc.pcm16_encode(chunk[i]))
            assert (g["started"], g["ended"], g["in_speech"], g["continued"]) == (0, 0, False, 0)


@pytest.mark.gpu
def test_wire_cfg5_scale(af, orc):
    """1024 streams x 20 ticks of 20 ms at 48 kHz, 80 mels + VAD, gated; 16 streams checked, the first and the last among them."""
    from audioflow import synth
    S, tick, n_ticks = 1024, 960, 20
    rng = np.random.default_rng(3)
    xs = np.stack([synth.stream(2000 + i, tick * n_ticks / 48000 + 0.01, 48000, 1)[: tick * n_ticks] for i in range(S)])
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=80)), S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    ses.enable_wire(gate=True)
    ticks = []
    for t in range(n_ticks):
        r = ses.push(xs[:, t * tick:(t + 1) * tick])
        w = ses.wire()
        w["n_frames"] = r["n_frames"]
        ticks.append(w)
    check = sorted({0, S - 1, *rng.choice(np.arange(1, S - 1), 14, replace=False).tolist()})
    assert len(check) == 16
    for i in check:
        ref_pcm = np.concatenate(_ref_pcm(orc, xs[i], 48000, 1, "f32", tick, n_ticks))
        states, _ = orc.VoiceActivityDetector().stream(ref_pcm, 400, 160)
        events, segs = _oracle_events(orc, states, [w["n_frames"] for w in ticks], 160)
        want = orc.pcm16_encode(orc.vad_gate(ref_pcm, None, segs, 160)[0])
        assert np.array_equal(np.concatenate([w["streams"][i]["pcm16"] for w in ticks]), want), i
        for w, ev in zip(ticks, events):
            g = w["streams"][i]
            assert (w["first_frame"], g["started"], g["ended"], g["in_speech"], g["continued"], g["n_samples"]) == ev, i
            assert g["base64"] == _b64(g["pcm16"])


@pytest.mark.gpu
def test_wire_off_means_off(af, orc):
    """Enabled-then-disabled and never-enabled sessions launch the same kernels and compute the same; on adds one launch."""
    from audioflow import synth
    S, tick, n_ticks = 8, 960, 12
    xs = np.stack([synth.stream(500 + i, tick * n_ticks / 48000 + 0.01, 48000, 1)[: tick * n_ticks] for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    never, off, on = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(3))
    off.enable_wire(gate=True)
    off.enable_wire(None)
    on.enable_wire(gate=True)
    with pytest.raises(ValueError):
        off.wire()
    for t in range(n_ticks):
        x = xs[:, t * tick:(t + 1) * tick]
        res, launches = [], []
        for ses in (never, off, on):
            l0 = af.kernel_launch_count()
            res.append(ses.push(x))
            launches.append(af.kernel_launch_count() - l0)
        assert launches[0] == launches[1] and launches[2] == launches[0] + 1, launches
        for k in ("pcm", "logmel", "vad"):
            assert np.array_equal(res[0][k], res[1][k]) and np.array_equal(res[0][k], res[2][k]), k


@pytest.mark.gpu
def test_wire_errors(af, orc):
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False)), 2, 48000, 1, af.AF_FMT_F32, max_tick_samples=960)
    with pytest.raises(ValueError):
        ses.enable_wire(gate=True)                                  # gating needs the VAD
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=0, vad_frame_len=160, vad_hop=320)), 2, 48000, 1, af.AF_FMT_F32,
                     max_tick_samples=960)
    with pytest.raises(ValueError):
        ses.enable_wire(gate=True)                                  # a hop longer than its frame is not there when it completes
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=80)), 2, 48000, 1, af.AF_FMT_F32, max_tick_samples=960)
    with pytest.raises(ValueError):
        ses.enable_wire(gate=True, mem=7)
    with pytest.raises(ValueError):
        ses.enable_wire(gate=False, pcm16=False, base64=False)
    ses.enable_wire(gate=True)
    with pytest.raises(ValueError):
        ses.wire()                                                  # nothing pushed since enabling
    ses.push(np.zeros((2, 960), np.float32))
    w = ses.wire()
    assert all(s["n_samples"] == 0 and s["base64"] == b"" for s in w["streams"])
    ses.enable_wire(gate=False, base64=False)
    with pytest.raises(ValueError):
        ses.wire()
    r = ses.push(np.zeros((2, 960), np.float32))
    w = ses.wire()
    assert all(s["n_samples"] == r["pcm"].shape[1] > 0 and s["base64"] is None and s["n_chars"] == 0 for s in w["streams"])
    assert all(np.array_equal(s["pcm16"], np.zeros(r["pcm"].shape[1], np.int16)) for s in w["streams"])


# ---------------------------------------------------------------------------------------------------------------------
def test_wire_abi_layout(tmp_path):
    """af_wire_config / af_wire_tick as a C compiler lays them out == the ctypes mirror; the Rust mirror declares the same
    fields in the same order."""
    import audioflow as af
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "audioflow_gpu.h"\n'
                   "#define F(t, f) printf(#t \" \" #f \" %zu %zu\\n\", offsetof(t, f), sizeof(((t *)0)->f));\n"
                   "int main(void) {\n"
                   '  printf("af_wire_config size %zu\\n", sizeof(af_wire_config));\n'
                   '  printf("af_wire_tick size %zu\\n", sizeof(af_wire_tick));\n'
                   "  F(af_wire_config, gate) F(af_wire_config, pcm16) F(af_wire_config, base64) F(af_wire_config, mem)\n"
                   "  F(af_wire_tick, n_samples) F(af_wire_tick, n_chars) F(af_wire_tick, continued) F(af_wire_tick, started)\n"
                   "  F(af_wire_tick, ended) F(af_wire_tick, in_speech) F(af_wire_tick, pad)\n"
                   "  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    lines = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split("\n")
    structs = {"af_wire_config": af.WireConfigC, "af_wire_tick": af.WireTickC}
    for ln in filter(None, lines):
        name, field, a, *b = ln.split()
        cs = structs[name]
        if field == "size":
            assert C.sizeof(cs) == int(a), name
        else:
            assert getattr(cs, field).offset == int(a) and getattr(cs, field).size == int(b[0]), (name, field)
    ffi = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "ffi.rs")).read()
    for name, cs in structs.items():
        m = re.search(r"pub struct %s \{(.*?)\}" % name, ffi, re.S)
        assert m, f"ffi.rs has no {name}"
        assert re.findall(r"pub (\w+):", m.group(1)) == [f for f, _ in cs._fields_], name
