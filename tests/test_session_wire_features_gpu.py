"""Wire features of sessions (af_session_enable_wire_features / af_session_wire_features): beside the gated wire payload,
per tick and stream the log-mel rows of exactly the frames the payload keeps.  Every tick, every stream: the rows are, bit
for bit, the kept frames' rows of the same tick's log-mel output, the kept frames follow the wire's rule (Speech, or the
Ending frame after Speech, across ticks), their count times the hop is the payload's n_samples, and the front `continued /
hop` rows are the tick's first frames.  Over a stream's life the rows concatenate to orc_vad_gate's log-mel over the
session's own concatenated log-mel and states (bitwise) and over the oracle's log-mel of its PCM (within
assert_logmel_close).  Checked streams are also compared bitwise against one-stream twin sessions fed the same ticks."""
import ctypes as C
import os
import re
import types

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal, assert_logmel_close
from test_session_streams_gpu import _source
from test_session_wire_gpu import _device_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPEECH, ENDING, HOP = 1, 2, 160


def _kept(states, prev):
    """The frames the gated wire keeps: Speech, or Ending right after Speech (prev: the state before the first frame)."""
    st = np.asarray(states, np.uint8)
    pre = np.concatenate([np.array([prev], np.uint8), st[:-1]])
    return np.nonzero((st == SPEECH) | ((st == ENDING) & (pre == SPEECH)))[0]


def _features(ses):
    """(per-stream [n_frames, n_mels] rows, n_frames) of the last push, device rows copied to the host."""
    import audioflow as af
    rows, n = ses.wire_features()
    if ses.features_mem == af.AF_MEM_DEVICE:                     # (pointer, stride in floats)
        ptr, stride = rows
        M = ses.pipe.cfg.n_mels
        all_rows = _device_rows(ptr, ses.S, stride, np.float32)
        rows = [all_rows[k, :int(n[k]) * M].reshape(-1, M).copy() for k in range(ses.S)]
    return rows, n


class _Life:
    def __init__(self):
        self.pcm, self.lm, self.vad, self.feat = [], [], [], []


class Driver:
    """A session of `formats` with the gated wire and its features on, pushed ragged ticks from per-stream sources.  Every
    tick checks every stream against its own tick outputs; streams in `twins` are also compared with one-stream twin
    sessions; a life (start to end, reset or restart) is checked whole when it closes."""

    def __init__(self, af, orc, pipe, formats, stream_format, mem, twins=(), seconds=6.0, source=None):
        self.af, self.orc, self.pipe, self.formats, self.seconds = af, orc, pipe, formats, seconds
        self.M = pipe.cfg.n_mels
        self.ses = af.Session.formats(pipe, formats, stream_format)
        self.ses.enable_wire(gate=True, mem=af.AF_MEM_HOST)
        self.ses.enable_wire_features(True, mem)
        self.S = self.ses.S
        self.source = source or (lambda k, rate, ch: _source(orc, 500 + 7 * k, seconds, rate, ch, "f32"))
        self.src = [self.source(k, *formats[f][:2]) for k, f in enumerate(stream_format)]
        self.cur = [0] * self.S
        self.prev = [0] * self.S
        self.life = [_Life() for _ in range(self.S)]
        self.twin = {}
        for k in twins:
            t = af.Session.formats(pipe, formats, [int(stream_format[k])])
            t.enable_wire(gate=True, mem=af.AF_MEM_HOST)
            t.enable_wire_features(True, af.AF_MEM_HOST)
            self.twin[k] = t
        self.closed = self.closed_open = 0

    def ch(self, k):
        return self.formats[self.ses.stream_format[k]][1]

    def max_frames(self, k):
        r, c, m = self.formats[self.ses.stream_format[k]]
        return m // c

    def samples(self, k, frames):
        n = frames * self.ch(k)
        if self.cur[k] + n > len(self.src[k]):
            self.cur[k] = 0
        x = self.src[k][self.cur[k]:self.cur[k] + n]
        self.cur[k] += n
        return x

    def ragged(self, rng):
        counts = []
        for k in range(self.S):
            m, pick = self.max_frames(k), int(rng.integers(0, 6))
            counts.append(0 if pick == 0 else 1 if pick == 1 else m if pick == 2 else int(rng.integers(0, m + 1)))
        return counts

    def tick(self, frames, end=None):
        end = [False] * self.S if end is None else [bool(e) for e in end]
        xs = [self.samples(k, n) for k, n in enumerate(frames)]
        r = self.ses.push_streams(xs, end)
        w = self.ses.wire()
        rows, n = _features(self.ses)
        for k in range(self.S):
            st, lm, g = r["vad"][k], r["logmel"][k], w["streams"][k]
            kept = _kept(st, self.prev[k])
            assert int(n[k]) == len(kept) and int(n[k]) * HOP == g["n_samples"], (k, int(n[k]), len(kept), g["n_samples"])
            assert_bit_equal(rows[k], lm[kept], f"stream {k} feature rows")
            c = g["continued"] // HOP
            assert list(kept[:c]) == list(range(c)), (k, c, kept[:c])
            L = self.life[k]
            L.pcm.append(r["pcm"][k]); L.lm.append(lm); L.vad.append(st); L.feat.append(rows[k])
            if len(st):
                self.prev[k] = int(st[-1])
        for k, t in self.twin.items():
            rt = t.push_streams([xs[k]], [end[k]])
            tr, tn = _features(t)
            assert_bit_equal(rt["logmel"][0], r["logmel"][k], f"stream {k} log-mel vs its twin")
            assert int(tn[0]) == int(n[k]), k
            assert_bit_equal(tr[0], rows[k], f"stream {k} feature rows vs its twin")
            tw = t.wire()["streams"][0]
            assert {q: v for q, v in tw.items() if q != "pcm16"} == {q: v for q, v in w["streams"][k].items() if q != "pcm16"}, k
        for k in range(self.S):
            if end[k]:
                self.closed_open += self.prev[k] == SPEECH              # the end closed an open segment
                self.close(k)
        return r

    def close(self, k):
        """Stream k's life is over: its feature rows concatenate to orc_vad_gate's log-mel."""
        L = self.life[k]
        if L.vad:
            st = np.concatenate(L.vad)
            lm = np.concatenate(L.lm).reshape(-1, self.M)
            pcm = np.concatenate(L.pcm)
            got = np.concatenate(L.feat).reshape(-1, self.M)
            segs = self.orc.vad_segments(st)
            assert_bit_equal(got, self.orc.vad_gate(None, lm, segs, HOP)[1], f"stream {k} features vs orc_vad_gate")
            ref = self.orc.logmel(pcm, self.orc.default_feat_config(self.M))
            assert_logmel_close(got, self.orc.vad_gate(None, ref, segs, HOP)[1], f"stream {k} features vs oracle log-mel")
        self.life[k] = _Life()
        self.prev[k] = 0
        self.closed += 1

    def reset(self, ids):
        self.ses.reset_streams(ids)
        for k in set(ids):
            if k in self.twin:
                self.twin[k].reset_streams([0])
            self.close(k)

    def restart(self, ids, fmts):
        self.ses.restart_streams(ids, fmts)
        for k, f in zip(ids, fmts):
            if k in self.twin:
                self.twin[k].restart_streams([0], [f])
            self.close(k)
            self.src[k] = self.source(k + 1000 * self.closed, *self.formats[f][:2])
            self.cur[k] = 0

    def set_vad_configs(self, ids, cfgs):
        self.ses.set_vad_configs(ids, cfgs)
        for k, c in zip(ids, cfgs):
            if k in self.twin:
                self.twin[k].set_vad_configs([0], [c])

    def finish(self):
        for k in range(self.S):
            self.close(k)


FORMATS = [(48000, 1, 960), (44100, 1, 882), (16000, 1, 320), (48000, 2, 1920)]


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_mels", [80, 128, 30])
@pytest.mark.parametrize("mem", ["host", "device"])
def test_rows_are_the_kept_frames_of_the_tick(af, orc, n_mels, mem):
    """Lockstep 20 ms and 200 ms ticks: per tick and stream the rows are the kept frames' rows of the tick's log-mel
    (n_mels = 30 takes the kernel's scalar path); over the whole run they are orc_vad_gate's log-mel."""
    m = af.AF_MEM_HOST if mem == "host" else af.AF_MEM_DEVICE
    pipe = af.Pipeline(af.pipeline_config(n_mels=n_mels, vad=af.VadConfig(silence_timeout_frames=3, min_speech_frames=2)))
    d = Driver(af, orc, pipe, [(48000, 1, 9600)], [0] * 6, m, twins=(0, 5), seconds=8.0)
    for t in range(40):
        d.tick([960 if t % 5 else 9600] * d.S)
    d.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("mem", ["host", "device"])
def test_ragged_mixed_formats_restarts_and_vad_configs(af, orc, mem):
    """12 streams in four capture formats (44.1 kHz and stereo among them), ragged ticks, ends, reset_streams,
    restart_streams into another format, per-stream VAD configurations set at the start and changed mid-stream; six
    streams have one-stream twins."""
    m = af.AF_MEM_HOST if mem == "host" else af.AF_MEM_DEVICE
    rng = np.random.default_rng(7 + m)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    sf = [k % len(FORMATS) for k in range(12)]
    d = Driver(af, orc, pipe, FORMATS, sf, m, twins=(0, 1, 2, 3, 6, 11))
    V = af.VadConfig
    d.set_vad_configs([1, 2, 6], [V(threshold_db=-40.0, min_speech_frames=1), V(smoothing_factor=0.6, silence_timeout_frames=4),
                                  V(threshold_db=-55.0, silence_timeout_frames=2)])
    for t in range(60):
        end = [bool(rng.random() < 0.04) for _ in range(d.S)]
        d.tick(d.ragged(rng), end)
        if t == 20:
            d.reset([3, 4])
        if t == 30:
            d.restart([0, 6, 7], [1, 3, 2])
        if t == 35:
            d.set_vad_configs([0, 11], [V(threshold_db=-35.0, min_speech_frames=4), V(silence_timeout_frames=1)])
        if t == 45:
            d.restart([1], [0])
    assert d.closed >= 8
    d.finish()


def _tone(seconds, rate, ch, freq=440.0):
    """A loud steady tone: the detector stays in Speech, so an end closes an open segment.  A noise floor keeps every mel
    band off the log floor (a pure tone's empty bands put the relative L2 of any f32 path beyond the log-mel tolerance)."""
    t = np.arange(int(seconds * rate)) / rate
    noise = np.random.default_rng(int(freq)).normal(0.0, 0.01, t.size)
    x = (0.3 * np.sin(2 * np.pi * freq * t) + noise).astype(np.float32)
    return np.repeat(x, ch) if ch > 1 else x


@pytest.mark.gpu
@pytest.mark.parametrize("residual", [0, 127])
def test_ends_close_open_segments(af, orc, residual):
    """Streams end with `residual` frames left before the flush, in Speech (tone) or in bursts; their next lives start
    afresh.  The end's tick keeps its last Speech frames and the next life opens no segment it did not start."""
    rng = np.random.default_rng(residual)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    src = lambda k, rate, ch: _tone(6.0, rate, ch, 300 + 50 * k) if k % 2 == 0 else _source(orc, 40 + k, 6.0, rate, ch, "f32")
    d = Driver(af, orc, pipe, [(48000, 1, 960), (44100, 1, 882)], [0, 0, 1, 1], af.AF_MEM_HOST, twins=(0, 2, 3), source=src)
    total = [0] * d.S
    for t in range(48):
        frames, end = [], []
        for k in range(d.S):
            mx = d.max_frames(k)
            n = int(rng.integers(mx // 2, mx + 1))
            last = t % 12 == 11
            if last:                                         # the frames pushed in this life leave `residual` behind
                n = (residual - total[k]) % 128 + 128 * ((mx - (residual - total[k]) % 128) // 128)
            frames.append(n)
            end.append(last)
            total[k] = 0 if last else total[k] + n
        d.tick(frames, end)
    assert d.closed == 4 * d.S and d.closed_open >= 4
    d.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("dst_mem", ["host", "device"])
def test_moved_caller_continues_its_segment(af, orc, dst_mem):
    """A caller in the middle of an utterance is exported from session A and imported into session B (other size, other
    format list, features on): its rows go on exactly as those of a never-moved twin, the segment open at the move
    included.  B's query refuses between the import and its next push."""
    m = af.AF_MEM_HOST if dst_mem == "host" else af.AF_MEM_DEVICE
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    rate, tick = 44100, 882
    x = _tone(4.0, rate, 1)
    x[int(2.5 * rate):] *= 0.0                                    # the utterance ends after the move: the segment closes in B
    a = af.Session(pipe, 4, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session.formats(pipe, [(16000, 1, 320), (rate, 1, 2 * tick)], [0] * 6)
    twin = af.Session(pipe, 1, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    for s, fm in ((a, af.AF_MEM_HOST), (b, m), (twin, af.AF_MEM_HOST)):
        s.enable_wire(gate=True)
        s.enable_wire_features(True, fm)
    slot_a, slot_b = 2, 4
    empty = np.zeros(0, np.float32)
    moved, continued = False, 0
    for t in range(150):
        chunk = x[t * tick:(t + 1) * tick]
        if not moved:
            b.push_streams([empty] * b.S)
            b.wire_features()                                    # valid before the import
        rt = twin.push_streams([chunk])
        tr, tn = _features(twin)
        ses, slot = (b, slot_b) if moved else (a, slot_a)
        r = ses.push_streams([chunk if k == slot else empty for k in range(ses.S)])
        rows, n = _features(ses)
        assert int(n[slot]) == int(tn[0]), t
        assert_bit_equal(rows[slot], tr[0], f"tick {t} rows")
        assert_bit_equal(r["logmel"][slot], rt["logmel"][0], f"tick {t} log-mel")
        if moved:
            continued += ses.wire()["streams"][slot]["continued"]
        if t == 60:
            assert twin.wire()["streams"][0]["in_speech"]           # mid-utterance
            rec = a.export_streams([slot_a])
            b.import_streams([slot_b], rec)
            a.reset_streams([slot_a])
            with pytest.raises(ValueError):
                b.wire_features()
            rc = af.load_library().af_session_wire_features(b._h, None, None, None)
            assert rc == af.AF_ERR_INVALID
            moved = True
    assert continued > 0


@pytest.mark.gpu
def test_cfg5_scale_and_launches(af, orc):
    """1024 streams x 20 ms at 48 kHz, 80 mels, VAD on, gated wire: with features off the lockstep tick launches what it
    launches without them; on, exactly one kernel more.  16 streams checked per tick, the first and the last among them."""
    from audioflow import synth
    S, tick, n_ticks = 1024, 960, 24
    rng = np.random.default_rng(5)
    xs = np.stack([synth.stream(4000 + i, tick * n_ticks / 48000 + 0.01, 48000, 1)[: tick * n_ticks] for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    off, on = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
    for s in (off, on):
        s.enable_wire(gate=True)
    on.enable_wire_features(True, af.AF_MEM_DEVICE)
    check = sorted({0, S - 1, *rng.choice(np.arange(1, S - 1), 14, replace=False).tolist()})
    prev = np.zeros(S, np.uint8)
    for t in range(n_ticks):
        x = xs[:, t * tick:(t + 1) * tick]
        l0 = af.kernel_launch_count()
        ro = off.push(x)
        l1 = af.kernel_launch_count()
        r = on.push(x)
        l2 = af.kernel_launch_count()
        if t > 0:
            assert l1 - l0 == 5, l1 - l0                             # ingest+resample, fused (2), scan, wire
        assert l2 - l1 == l1 - l0 + 1, (l1 - l0, l2 - l1)
        assert_bit_equal(ro["logmel"], r["logmel"]); assert_bit_equal(ro["vad"], r["vad"])
        rows, n = _features(on)
        w = on.wire()["streams"]
        for k in check:
            kept = _kept(r["vad"][k], prev[k])
            assert int(n[k]) == len(kept) and int(n[k]) * HOP == w[k]["n_samples"], k
            assert_bit_equal(rows[k], r["logmel"][k][kept], f"tick {t} stream {k}")
        assert (n.astype(np.int64) * HOP == np.array([g["n_samples"] for g in w])).all()
        if r["n_frames"]:
            prev = r["vad"][:, -1].copy()


@pytest.mark.gpu
@pytest.mark.parametrize("wire_mem", ["host", "device"])
def test_off_means_off(af, orc, wire_mem):
    """A session that never enabled the features, one that enabled and disabled them, and one whose wire was turned off
    and on again compute the same bits with the same launches; allocations return to their baseline after disable and
    destroy."""
    from audioflow import synth
    m = af.AF_MEM_HOST if wire_mem == "host" else af.AF_MEM_DEVICE
    S, tick, n_ticks = 8, 960, 10
    xs = np.stack([synth.stream(700 + i, tick * n_ticks / 48000 + 0.01, 48000, 1)[: tick * n_ticks] for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    warm = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)   # the pipeline's and the context's buffers
    warm.push(xs[:, :tick])
    del warm
    base = af.live_allocations()
    never, disabled, rewired = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(3))
    for s in (never, disabled, rewired):
        s.enable_wire(gate=True, mem=m)
        s.push(xs[:, :tick])
    held = af.live_allocations()
    disabled.enable_wire_features(True, m)
    assert af.live_allocations()[0] > held[0]
    disabled.enable_wire_features(False)
    assert af.live_allocations() == held                             # the first tick completed no frame: nothing staged yet
    # once ticks complete frames (and the staging the caller's log-mel needs exists), a tick with features on allocates
    # nothing, and disabling returns to the count before enabling
    for s in (never, disabled, rewired):
        s.push(xs[:, tick:2 * tick])
    held = af.live_allocations()
    disabled.enable_wire_features(True, m)
    on = af.live_allocations()
    for s in (never, disabled, rewired):
        s.push(xs[:, 2 * tick:3 * tick])
    assert int(disabled.wire_features()[1].size) == S and af.live_allocations() == on
    disabled.enable_wire_features(False)
    assert af.live_allocations() == held
    rewired.enable_wire_features(True, m)
    rewired.enable_wire(gate=True, mem=m)                            # a new wire configuration turns the features off
    assert af.live_allocations() == held
    for s in (disabled, rewired):
        with pytest.raises(ValueError):
            s.wire_features()
    for t in range(3, n_ticks):
        x = xs[:, t * tick:(t + 1) * tick]
        res, launches, wires = [], [], []
        for s in (never, disabled, rewired):
            l0 = af.kernel_launch_count()
            res.append(s.push(x))
            launches.append(af.kernel_launch_count() - l0)
            wires.append(s.wire())
        assert launches[0] == launches[1] == launches[2], launches
        for k in ("pcm", "logmel", "vad"):
            assert_bit_equal(res[0][k], res[1][k], k); assert_bit_equal(res[0][k], res[2][k], k)
        for a_, b_, c_ in zip(*(w["streams"] for w in wires)):
            assert {q: v for q, v in a_.items() if q not in ("pcm16",)} == {q: v for q, v in b_.items() if q not in ("pcm16",)}
            assert {q: v for q, v in a_.items() if q not in ("pcm16",)} == {q: v for q, v in c_.items() if q not in ("pcm16",)}
    # the wire turned off turns the features off; re-enabling the wire does not bring them back
    disabled.enable_wire_features(True, m)
    disabled.enable_wire(None)
    assert af.live_allocations()[0] < held[0]
    with pytest.raises(ValueError):
        disabled.wire_features()
    del never, disabled, rewired, s
    assert af.live_allocations() == base


@pytest.mark.gpu
def test_refusals_leave_the_session_untouched(af, orc):
    """Each refusal is AF_ERR_INVALID and changes nothing: a session that met them computes, bit for bit, what a twin
    that never did computes."""
    from audioflow import synth
    L = af.load_library()
    H, D = af.AF_MEM_HOST, af.AF_MEM_DEVICE
    en = lambda s, on, mem: L.af_session_enable_wire_features(s._h, on, mem)
    # sessions that cannot have features
    no_mels = af.Session(af.Pipeline(af.pipeline_config(n_mels=0)), 2, 48000, 1, af.AF_FMT_F32, max_tick_samples=960)
    no_mels.enable_wire(gate=True)
    assert en(no_mels, 1, H) == af.AF_ERR_INVALID                 # n_mels == 0
    no_vad = af.Session(af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=False)), 2, 48000, 1, af.AF_FMT_F32,
                        max_tick_samples=960)
    no_vad.enable_wire(gate=False)
    assert en(no_vad, 1, H) == af.AF_ERR_INVALID                  # vad_enable == 0 (and so no gated wire)
    vad20 = af.Session(af.Pipeline(af.pipeline_config(n_mels=0, vad_frame_len=320, vad_hop=320)), 2, 48000, 1, af.AF_FMT_F32,
                       max_tick_samples=960)
    vad20.enable_wire(gate=True)
    assert en(vad20, 1, H) == af.AF_ERR_INVALID                   # 20 ms VAD frames (a session refuses them with n_mels)
    # a session that can, against its twin
    S, tick = 4, 960
    xs = np.stack([synth.stream(900 + i, 1.0, 48000, 1)[: tick * 30] for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    ses, twin = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
    assert en(ses, 1, H) == af.AF_ERR_INVALID                     # the wire is off
    ses.enable_wire(gate=False)
    assert en(ses, 1, H) == af.AF_ERR_INVALID                     # the wire is not gated
    for s in (ses, twin):
        s.enable_wire(gate=True)
    assert en(ses, 1, 7) == af.AF_ERR_INVALID                     # a bad mem
    with pytest.raises(ValueError):
        ses.wire_features()                                       # the features are off
    for s in (ses, twin):
        s.enable_wire_features(True, D)
        with pytest.raises(ValueError):
            s.wire_features()                                     # nothing pushed since enabling
    for t in range(30):
        x = xs[:, t * tick:(t + 1) * tick]
        r1, r2 = ses.push(x), twin.push(x)
        if t == 10:
            assert en(ses, 1, 7) == af.AF_ERR_INVALID             # refused while on: the rows stay on and valid
            assert L.af_session_wire_features(ses._h, None, None, None) == af.AF_OK
        if t == 20:
            assert en(ses, 1, -1) == af.AF_ERR_INVALID
        (f1, n1), (f2, n2) = _features(ses), _features(twin)
        assert np.array_equal(n1, n2), t
        for k in range(S):
            assert_bit_equal(f1[k], f2[k], f"tick {t} stream {k}")
        assert_bit_equal(r1["logmel"], r2["logmel"]); assert_bit_equal(r1["vad"], r2["vad"])
    assert L.af_session_wire_features(None, None, None, None) == af.AF_ERR_INVALID
    assert L.af_session_enable_wire_features(None, 1, H) == af.AF_ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
def _no_library():
    raise AssertionError("the library was called")


def test_python_arguments_are_checked_before_the_library(monkeypatch):
    """No GPU: enable_wire_features refuses a bad mem, a session without the gated wire, a pipeline without log-mel or
    VAD, and 20 ms VAD frames before it calls the library."""
    import audioflow as af
    monkeypatch.setattr(af, "load_library", _no_library)

    def session(wire_mem=af.AF_MEM_HOST, gate=True, **cfg):
        c = af.PipelineConfigC(n_mels=80, vad_enable=1)
        for k, v in cfg.items():
            setattr(c, k, v)
        s = af.Session.__new__(af.Session)
        s.pipe, s._h, s.S = types.SimpleNamespace(cfg=c), None, 2
        s.wire_mem, s.wire_gate, s.features_mem = wire_mem, gate, None
        return s

    for s, mem in ((session(), 7), (session(), -1), (session(wire_mem=None), af.AF_MEM_HOST),
                   (session(gate=False), af.AF_MEM_HOST), (session(n_mels=0), af.AF_MEM_DEVICE),
                   (session(vad_enable=0), af.AF_MEM_HOST), (session(vad_frame_len=320, vad_hop=320), af.AF_MEM_HOST)):
        with pytest.raises(ValueError):
            s.enable_wire_features(True, mem)
    for cfg in (dict(), dict(vad_frame_len=400, vad_hop=160)):      # accepted: the call reaches the library
        with pytest.raises(AssertionError):
            session(**cfg).enable_wire_features(True, af.AF_MEM_DEVICE)


def test_new_symbols_in_every_mirror():
    """The two calls are declared in the header, exported by the library, bound by ctypes, the C++ mirror and the Rust
    shim."""
    import audioflow as af
    names = ("af_session_enable_wire_features", "af_session_wire_features")
    header = open(os.path.join(ROOT, "include", "audioflow_gpu.h")).read()
    hpp = open(os.path.join(ROOT, "audio-flow-rs_b200", "host", "audioflow.hpp")).read()
    ffi = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "ffi.rs")).read()
    L = af.load_library()
    for n in names:
        assert re.search(r"AF_API\s+int\s+%s\s*\(" % n, header), n
        assert getattr(L, n).restype is C.c_int, n
        assert n + "(" in hpp, n
        assert re.search(r"pub fn %s\s*\(" % n, ffi), n
