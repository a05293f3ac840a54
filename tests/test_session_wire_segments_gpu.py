"""Segment table of the gated session wire (af_session_enable_wire_segments / af_session_wire_segments): per stream and
tick, the pieces of every segment in the tick's gated payload.

Every tick and every checked stream: the per-tick rules of the header (pieces tile the payload, CONTINUED / CLOSED against
the af_wire_tick counts, the closing-only piece), the PCM16 payload and the wire feature rows of each piece are the
stream's own samples and log-mel rows of the piece's frames, and -- whole-life equality -- the pieces since the stream's
origin, joined and made global with af_session_wire_first_frames, are orc_vad_segments pre-rolled by segments_preroll
(clamped at the origin), with orc_vad_gate's segment offsets."""
import ctypes as C
import gc
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal
from test_session_wire_gpu import _device_rows
from test_session_wire_preroll_gpu import Driver, _bursts, _rows, _payloads, _strip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CONT, CLOSED = 1, 2


def segments_preroll(seg, P):
    """The pre-roll rule: segment k [start, end) starts at max(start - P, end of segment k - 1, 0); ends are kept."""
    out = np.array(seg, np.int64).reshape(-1, 2)
    for k in range(len(out)):
        out[k, 0] = max(out[k, 0] - P, out[k - 1, 1] if k else 0, 0)
    return out


def _table(ses):
    """The segment table of the last push as per-stream WIRE_SEGMENT_DTYPE arrays (device rows copied to the host)."""
    import audioflow as af
    rows, n = ses.wire_segments()
    if ses.segments_mem == af.AF_MEM_DEVICE:
        ptr, stride = rows
        raw = _device_rows(ptr, ses.S, stride * 16, np.uint8)
        rows = [raw[k, :int(n[k]) * 16].copy().view(af.WIRE_SEGMENT_DTYPE) for k in range(ses.S)]
    return rows, n


class SegLife:
    """One stream since its start: its states, PCM and log-mel, and the segments its pieces built since its origin."""

    def __init__(self, P, hop):
        self.P, self.hop = P, hop
        self.vad, self.pcm, self.lm = [], [], []
        self.n = 0                                        # frames since the start
        self.origin, self.closed, self.open, self.paid = 0, [], None, 0
        self.seen = dict(cont=0, closing_only=0, closing_only_empty=0, negative=0, preroll=0, multi=0, most=0)

    def new_origin(self, P=None):
        self.P = self.P if P is None else P
        self.origin, self.closed, self.paid = self.n, [], 0
        if self.open is not None:                         # an open segment carries on, clamped at the origin
            self.open = [self.n, self.n, None, 0]

    def tick(self, orc, segs, g, ff, vad, pcm=None, lm=None, pay=None, feat=None):
        """Checks one tick's pieces `segs` against the record g (a wire() stream dict), then the whole life."""
        hop, T = self.hop, len(vad)
        assert ff == self.n, (ff, self.n)
        segs = np.asarray(segs)
        n = len(segs)
        fl, nf, off = segs["flags"].astype(int), segs["n_frames"].astype(int), segs["offset"].astype(int)
        # per-tick rules
        assert (segs["pad"] == 0).all() and ((fl & ~3) == 0).all()
        assert n == 0 or off[0] == 0
        assert np.array_equal(off[1:], (off + nf)[:-1]), segs
        assert int(nf.sum()) * hop == g["n_samples"], (segs, g)
        assert int((fl & CONT == 0).sum()) == g["started"] and int((fl & CLOSED != 0).sum()) == g["ended"], (segs, g)
        assert not (fl[1:] & CONT).any()
        assert (nf[0] * hop if n and fl[0] & CONT else 0) == g["continued"], (segs, g)
        assert (fl[:-1] & CLOSED).all()
        assert n == 0 or bool(fl[-1] & CLOSED) == (not g["in_speech"]), (segs, g)
        assert n <= (T + 1) // 2 + 1
        for i, s in enumerate(segs):
            if nf[i] == 0:
                assert i == 0 and fl[i] == CONT | CLOSED and s["frame"] == 0, segs
            if fl[i] & CONT:
                assert s["frame"] == 0 and s["preroll"] == 0
            else:
                assert -self.P <= s["frame"] and 0 <= s["frame"] + s["preroll"] < T and s["preroll"] < nf[i], segs
        # the piece's payload samples and feature rows are the stream's own, frame for frame
        if pcm is not None:
            self.pcm.append(np.asarray(pcm, np.float32))
        if lm is not None and T:
            self.lm.append(np.asarray(lm, np.float32).reshape(T, -1))
        allp = np.concatenate(self.pcm) if self.pcm else None
        alll = np.concatenate(self.lm) if self.lm else None
        for s in segs:
            a, b = ff + int(s["frame"]), ff + int(s["frame"]) + int(s["n_frames"])
            o = int(s["offset"])
            if pay is not None and allp is not None:
                src = np.zeros((b - a) * hop, np.float32)
                part = allp[a * hop:b * hop]
                src[:len(part)] = part
                assert np.array_equal(pay[o * hop:(o + b - a) * hop], orc.pcm16_encode(src)), (s, a, b)
            if feat is not None:
                assert_bit_equal(feat[o:o + b - a], alll[a:b], f"feature rows of piece {s}")
        # join the pieces
        for i, s in enumerate(segs):
            a = ff + int(s["frame"])
            if fl[i] & CONT:
                assert self.open is not None and self.open[1] == a, (self.open, a)
                self.open[1] = a + int(nf[i])
                self.seen["cont"] += 1
            else:
                assert self.open is None, self.open
                self.open = [a, a + int(nf[i]), a + int(s["preroll"]), self.paid + int(s["offset"])]
                self.seen["negative"] += s["frame"] < 0
                self.seen["preroll"] += s["preroll"] > 0
            if nf[i] == 0:
                self.seen["closing_only"] += 1
                self.seen["closing_only_empty"] += T == 0
            if fl[i] & CLOSED:
                self.closed.append(self.open)
                self.open = None
        self.seen["multi"] += g["started"] >= 3
        self.seen["most"] = max(self.seen["most"], n)
        self.paid += int(nf.sum())
        self.vad.append(np.asarray(vad, np.uint8))
        self.n += T
        # whole-life equality
        st = np.concatenate(self.vad)
        raw = orc.vad_segments(st).astype(np.int64).reshape(-1, 2)
        ext = segments_preroll(raw, self.P)
        keep = ext[:, 1] > self.origin
        exp = np.array([[max(a, self.origin), b] for a, b in ext[keep]], np.int64).reshape(-1, 2)
        got = self.closed + ([self.open] if self.open is not None else [])
        assert np.array_equal(np.array([[a, b] for a, b, _, _ in got], np.int64).reshape(-1, 2), exp), (got[-3:], exp[-3:])
        for (_, _, onset, _), r in zip(got, raw[keep]):
            assert onset is None or onset == r[0], (onset, r)
        _, _, goff = orc.vad_gate(None, None, exp.astype(np.uint32), hop)
        assert [q for _, _, _, q in got] == [int(x) for x in goff[:-1]] and int(goff[-1]) == self.paid


class SegDriver(Driver):
    """The pre-roll tests' Driver (payloads, features, records against the oracle and twins) with the segment table on
    in `smem` rows; every tick also checks every checked stream's table (SegLife) and the twins' tables."""

    def __init__(self, af, orc, pipe, formats, stream_format, P, fmem=None, wmem=None, smem=None, **kw):
        super().__init__(af, orc, pipe, formats, stream_format, P, fmem, wmem, **kw)
        smem = af.AF_MEM_HOST if smem is None else smem
        for s in (self.ses, *self.twin.values()):
            s.enable_wire_segments(True, smem)
        self.seg = [SegLife(P, self.hop) for _ in range(self.S)]

    def tick(self, frames, end=None, lockstep=False):
        r = super().tick(frames, end, lockstep)
        end = [False] * self.S if end is None else end
        w = self.ses.wire()
        tab, _ = _table(self.ses)
        pays, _ = _payloads(self.ses, w)
        rows = _rows(self.ses)[0] if self.M else None
        for k in self.check:
            self.seg[k].tick(self.orc, tab[k], w["streams"][k], int(w["first_frames"][k]), r["vad"][k], r["pcm"][k],
                             r["logmel"][k] if self.M else None, pays[k], rows[k] if self.M else None)
        for k, t in self.twin.items():
            assert np.array_equal(_table(t)[0][0], tab[k]), f"stream {k} table vs its twin"
        for k in range(self.S):
            if end[k]:
                self.seg[k] = SegLife(self.P, self.hop)
        return r

    def reset(self, ids):
        super().reset(ids)
        for k in ids:
            self.seg[k] = SegLife(self.P, self.hop)

    def restart(self, ids, fmts):
        super().restart(ids, fmts)
        for k in ids:
            self.seg[k] = SegLife(self.P, self.hop)

    def set_preroll(self, P):
        super().set_preroll(P)
        for L in self.seg:
            L.new_origin(P)

    def seen(self, key):
        return sum(self.seg[k].seen[key] for k in self.check) if key != "most" else max(L.seen["most"] for L in self.seg)


def _vad(af, **kw):
    return af.VadConfig(**{"silence_timeout_frames": 2, "min_speech_frames": 1, **kw})


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [0, 30])
def test_20ms_ticks_synth(af, orc, P):
    """cfg5-like: lockstep 20 ms ticks at 48 kHz of the synth signal, 80 mels, features on (host rows)."""
    from audioflow import synth
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = SegDriver(af, orc, pipe, [(48000, 1, 960)], [0] * 6, P, af.AF_MEM_HOST)
    d.src = [synth.stream(k, 8.0, 48000) for k in range(d.S)]
    for t in range(300):
        d.tick([960] * d.S, lockstep=True)
    assert d.seen("cont") > 20 and sum(len(L.closed) for L in d.seg) >= 3


@pytest.mark.gpu
@pytest.mark.parametrize("P,smem", [(0, "host"), (0, "device"), (30, "device")])
def test_1s_ticks_several_utterances(af, orc, P, smem):
    """1 s ticks (48 kHz mono and 44.1 kHz stereo, synth and short bursts): ticks with three or more utterances, each a
    piece of its own."""
    from audioflow import synth
    m = af.AF_MEM_HOST if smem == "host" else af.AF_MEM_DEVICE
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = SegDriver(af, orc, pipe, [(48000, 1, 48000), (44100, 2, 88200)], [0, 1, 0, 1], P, af.AF_MEM_HOST, smem=m, twins=(1,))
    d.src[2] = synth.stream(2, 8.0, 48000)
    t48 = np.arange(48000 * 8) / 48000.0                 # 120 ms tones every 250 ms, a detector that follows them
    d.src[0] = (0.3 * np.sin(2 * np.pi * 440.0 * t48) * ((t48 % 0.25) < 0.12)).astype(np.float32)
    d.set_vad_configs([0], [af.VadConfig(smoothing_factor=0.9, silence_timeout_frames=2, min_speech_frames=1)])
    for t in range(7):
        d.tick([d.formats[f][2] // d.formats[f][1] for f in d.ses.stream_format])
    assert d.seen("multi") >= 1


def _alternating(frames, hop, loud, rng):
    """16 kHz mono whose VAD frame f (hop samples) is a loud tone when loud[f], else a faint noise floor."""
    x = rng.normal(0.0, 1e-4, frames * hop)
    t = np.arange(hop) / 16000.0
    for f in np.nonzero(loud)[0]:
        x[f * hop:(f + 1) * hop] += 0.5 * np.sin(2 * np.pi * 700.0 * t)
    return x.astype(np.float32)


@pytest.mark.gpu
def test_capacity_worst_case_and_sentinel(af, orc):
    """Alternating loud and quiet 20 ms frames, per-stream configurations whose smoothed energy follows each frame
    (smoothing 1.0), timeouts 0 and 1, min speech 0 and 2: as many segments per tick as the detector allows (min speech 2
    turns every quiet frame into Silence: one start every two frames).  Before every push the device rows are filled with
    a sentinel; after it, nothing past each stream's pieces was written, and the count stays within ceil(T / 2) + 1."""
    import torch
    hop, tick = 320, 320 * 40
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad=_vad(af), vad_frame_len=hop, vad_hop=hop))
    ses = af.Session(pipe, 4, 16000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    ses.enable_wire(gate=True, mem=af.AF_MEM_DEVICE)
    ses.enable_wire_segments(True, af.AF_MEM_DEVICE)
    V = af.VadConfig
    ses.set_vad_configs([0, 1, 2, 3], [V(threshold_db=-15.0, smoothing_factor=1.0, silence_timeout_frames=to, min_speech_frames=ms)
                                       for to, ms in ((0, 0), (1, 0), (0, 2), (1, 2))])
    rng = np.random.default_rng(4)
    n_fr = 40 * 30
    loud = np.arange(n_fr) % 2 == 0
    loud[200:260] = rng.random(60) < 0.5
    xs = np.stack([_alternating(n_fr, hop, np.roll(loud, k), rng) for k in range(4)])
    lives = [SegLife(0, hop) for _ in range(4)]
    SENT = 0xA5
    best = 0
    for t in range(30):
        sizes = [tick if t % 3 else int(rng.integers(1, 41)) * hop for _ in range(4)]
        if t:
            ptr, stride = ses.wire_segments()[0]

            class _Rows:
                __cuda_array_interface__ = {"shape": (4, stride * 16), "typestr": "|u1", "data": (ptr, False), "version": 2,
                                            "strides": None}
            torch.as_tensor(_Rows(), device="cuda").fill_(SENT)
            torch.cuda.synchronize()
        r = ses.push_streams([xs[k, (t * tick) % (n_fr * hop - tick):][:sizes[k]] for k in range(4)])
        (ptr, stride), n = ses.wire_segments()
        raw = _device_rows(ptr, 4, stride * 16, np.uint8)
        w = ses.wire()
        for k in range(4):
            T = len(r["vad"][k])
            assert int(n[k]) <= (T + 1) // 2 + 1 <= stride
            assert t == 0 or (raw[k, int(n[k]) * 16:] == SENT).all(), (t, k, int(n[k]))
            segs = raw[k, :int(n[k]) * 16].copy().view(af.WIRE_SEGMENT_DTYPE)
            lives[k].tick(orc, segs, w["streams"][k], int(w["first_frames"][k]), r["vad"][k])
            if T >= 10:
                best = max(best, int(n[k]) - (T + 1) // 2)
    assert best >= 0                                   # some tick held ceil(T / 2) starts (plus, at most, the open one)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [0, 7])
def test_closing_only_pieces(af, orc, P):
    """20 ms VAD frames, ticks of 1-3 frames: short bursts that never reach min speech close on a tick's first frame
    (Speech -> Silence), and streams that end mid-utterance -- with residual 0 and 127 of the 48 kHz resampler's 128-frame
    chunk, and with a last push of 0 samples -- close by the end; each such close is a CONTINUED | CLOSED piece of 0
    frames when the tick has no payload frame for it."""
    hop = 320
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad=_vad(af), vad_frame_len=hop, vad_hop=hop))
    ses = af.Session.formats(pipe, [(16000, 1, 3 * hop), (48000, 1, 9 * hop)], [0, 0, 1, 1])
    ses.enable_wire(gate=True)
    ses.enable_wire_segments(True, af.AF_MEM_HOST)
    if P:
        ses.set_wire_preroll(P)
    V = af.VadConfig
    ses.set_vad_configs([0, 1, 2, 3], [V(threshold_db=-30.0, smoothing_factor=1.0, silence_timeout_frames=1, min_speech_frames=5),
                                       V(threshold_db=-30.0, smoothing_factor=1.0, silence_timeout_frames=1, min_speech_frames=1),
                                       V(threshold_db=-30.0, smoothing_factor=1.0, silence_timeout_frames=3, min_speech_frames=1),
                                       V(threshold_db=-30.0, smoothing_factor=1.0, silence_timeout_frames=3, min_speech_frames=1)])
    rng = np.random.default_rng(9)
    loud16 = np.tile([0, 0, 0, 1, 1, 0, 0, 1, 1, 1, 0, 1, 1, 0, 0], 40).astype(bool)
    src = [_alternating(len(loud16), hop, loud16, rng)] * 2
    x48 = np.repeat(_alternating(len(loud16), hop, np.ones(len(loud16), bool), rng), 3)     # speech throughout
    src += [x48, x48]
    cur = [0] * 4
    lives = [SegLife(P, hop) for _ in range(4)]
    ends_seen = {0: 0, 127: 0, "empty": 0}
    for t in range(160):
        counts, end = [], []
        for k in range(4):
            if k < 2:
                counts.append(int(rng.integers(1, 4)) * hop); end.append(False)
            else:
                life_in = cur[k]
                phase = t % 8
                if phase == 7:                                    # the end: residual 0 or 127, or a push of 0 samples
                    kind = (0, 127, "empty")[(t // 8 + k) % 3]
                    if kind == "empty":
                        counts.append(0)
                    else:
                        counts.append((kind - life_in % 128) % 128 or 128)
                    end.append(True)
                    ends_seen[kind] += 1
                else:
                    counts.append(int(rng.integers(1, 10)) * 3 * hop // 3); end.append(False)
        xs = []
        for k in range(4):
            if cur[k] + counts[k] > len(src[k]):
                cur[k] = 0
            xs.append(src[k][cur[k]:cur[k] + counts[k]])
            cur[k] += counts[k]
        r = ses.push_streams(xs, end)
        w = ses.wire()
        tab, _ = _table(ses)
        for k in range(4):
            lives[k].tick(orc, tab[k], w["streams"][k], int(w["first_frames"][k]), r["vad"][k])
            if end[k]:
                assert w["streams"][k]["in_speech"] is False and (len(tab[k]) == 0 or tab[k][-1]["flags"] & CLOSED)
                lives[k] = SegLife(P, hop)
                cur[k] = 0
    assert min(ends_seen.values()) > 5
    # cur[] tracks input since each life's start: lives restart after an end
    co = sum(L.seen["closing_only"] for L in lives)
    assert co > 0


@pytest.mark.gpu
@pytest.mark.parametrize("P,mem", [(0, "host"), (12, "device")])
def test_ragged_mixed_formats_ends_resets_restarts(af, orc, P, mem):
    """12 streams in four capture formats (44.1 kHz stereo among them), ragged ticks, ends, reset_streams,
    restart_streams into another format, per-stream VAD configurations changed mid-stream; six streams have one-stream
    twins whose tables are the same."""
    m = af.AF_MEM_HOST if mem == "host" else af.AF_MEM_DEVICE
    rng = np.random.default_rng(21 + P)
    formats = [(48000, 1, 960), (44100, 2, 1764), (16000, 1, 320), (48000, 2, 1920)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = SegDriver(af, orc, pipe, formats, [k % 4 for k in range(12)], P, m, m, smem=m, twins=(0, 1, 2, 3, 6, 11))
    V = af.VadConfig
    d.set_vad_configs([1, 2, 6], [V(threshold_db=-40.0, min_speech_frames=1), V(smoothing_factor=0.6, silence_timeout_frames=4),
                                  V(threshold_db=-55.0, silence_timeout_frames=2)])
    for t in range(90):
        counts = []
        for k in range(d.S):
            ch = formats[d.ses.stream_format[k]][1]
            mx = formats[d.ses.stream_format[k]][2] // ch
            pick = int(rng.integers(0, 6))
            counts.append(0 if pick == 0 else 1 if pick == 1 else mx if pick == 2 else int(rng.integers(0, mx + 1)))
        d.tick(counts, [bool(rng.random() < 0.03) for _ in range(d.S)])
        if t == 25:
            d.reset([3, 4])
        if t == 40:
            d.restart([0, 6, 7], [1, 3, 2])
        if t == 50:
            d.set_vad_configs([0, 11], [V(threshold_db=-35.0, min_speech_frames=4), V(silence_timeout_frames=1)])
        if t == 65:
            d.restart([1], [0])
    assert d.seen("cont") > 10


@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 30, 100])
def test_preroll_pieces(af, orc, P):
    """20 ms ticks of short bursts: onsets within P frames of the previous close (the pieces become payload-adjacent),
    pre-rolls that reach into earlier pushes (frame < 0), and the pre-roll changed mid-stream (a new origin)."""
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = SegDriver(af, orc, pipe, [(48000, 1, 960)], [0] * 4, P, af.AF_MEM_DEVICE, af.AF_MEM_DEVICE, smem=af.AF_MEM_DEVICE,
                  twins=(2,))
    for t in range(200):
        if t == 120:
            d.set_preroll(max(1, P // 3))
        d.tick([960] * d.S, lockstep=True)
    assert d.seen("negative") > 0 and d.seen("preroll") > 5
    adjacent = sum(1 for L in d.seg for a, b in zip(L.closed, L.closed[1:]) if a[1] == b[0])
    assert adjacent > 0 or P == 1                      # (gaps of one frame are rare in this signal)


@pytest.mark.gpu
def test_vad_20ms_frames(af, orc):
    """VAD on 20 ms frames (vad_frame_len = vad_hop = 320), no log-mel, ragged ticks."""
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad=_vad(af), vad_frame_len=320, vad_hop=320))
    d = SegDriver(af, orc, pipe, [(48000, 1, 1920), (16000, 1, 640)], [0, 1, 0, 1], 0, None, hop=320, twins=(1,))
    rng = np.random.default_rng(3)
    for t in range(120):
        d.tick([int(rng.integers(0, d.formats[f][2] + 1)) for f in d.ses.stream_format])
    assert d.seen("cont") > 5


@pytest.mark.gpu
@pytest.mark.parametrize("P", [0, 25])
def test_import_continues_the_open_segment(af, orc, P):
    """A stream exported mid-utterance from session A and imported into session B: its first tick there starts with a
    CONTINUED piece, and the whole-life equality holds across the move (with a pre-roll, the import is an origin)."""
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    rate, tick = 44100, 882
    x = _bursts(78, 6.0, rate)
    a = af.Session(pipe, 4, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session.formats(pipe, [(16000, 1, 320), (rate, 1, 2 * tick)], [0] * 6)
    for s in (a, b):
        s.enable_wire(gate=True)
        s.enable_wire_features(True)
        s.set_wire_preroll(P)
        s.enable_wire_segments(True, af.AF_MEM_DEVICE if s is b else af.AF_MEM_HOST)
    slot_a, slot_b = 2, 4
    empty = np.zeros(0, np.float32)
    L = SegLife(P, 160)
    moved, first_after = False, None
    for t in range(250):
        chunk = x[t * tick:(t + 1) * tick]
        ses, slot = (b, slot_b) if moved else (a, slot_a)
        if not moved:
            b.push_streams([empty] * b.S)
        r = ses.push_streams([chunk if k == slot else empty for k in range(ses.S)])
        w = ses.wire()
        tab, _ = _table(ses)
        pays, _ = _payloads(ses, w)
        rows, _ = _rows(ses)
        L.tick(orc, tab[slot], w["streams"][slot], int(w["first_frames"][slot]), r["vad"][slot], r["pcm"][slot],
               r["logmel"][slot], pays[slot], rows[slot])
        if moved and first_after is None:
            first_after = tab[slot]
        if not moved and t >= 100 and w["streams"][slot]["in_speech"] and len(r["vad"][slot]):
            rec = a.export_streams([slot_a])
            b.import_streams([slot_b], rec)
            a.reset_streams([slot_a])
            if P:
                L.new_origin()
            moved = True
    assert moved and len(first_after) and first_after[0]["flags"] & CONT
    assert len(L.closed) >= 3


@pytest.mark.gpu
def test_host_and_device_rows_agree(af, orc):
    """The same ticks into a session with host rows and one with device rows: identical tables, P = 0 and P = 20."""
    S, tick = 5, 4800
    xs = np.stack([_bursts(50 + i, 6.0, 48000) for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    for P in (0, 20):
        h, d = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
        for s, m in ((h, af.AF_MEM_HOST), (d, af.AF_MEM_DEVICE)):
            s.enable_wire(gate=True, mem=m)
            s.set_wire_preroll(P)
            s.enable_wire_segments(True, m)
            assert s.wire_preroll == P                       # the table does not reset the pre-roll
        total = 0
        for t in range(60):
            x = xs[:, t * tick:(t + 1) * tick]
            h.push(x); d.push(x)
            (th, nh), (td, nd) = _table(h), _table(d)
            assert np.array_equal(nh, nd)
            for k in range(S):
                assert th[k].tobytes() == td[k].tobytes(), (P, t, k)
            total += int(nh.sum())
        assert total > 20


@pytest.mark.gpu
@pytest.mark.parametrize("P", [0, 30])
def test_1024_streams_table_off_is_unchanged(af, orc, P):
    """cfg5's shape (1024 x 20 ms at 48 kHz, 80 mels, VAD, gated wire with features on the device): with the table on
    (ticks 0-29) and off again (30-44) a session launches as many kernels per tick as one that never enabled it; payload
    bytes, af_wire_tick records and feature rows are identical; disabling releases exactly what enabling allocated; 16
    streams' tables are checked against the oracle."""
    S, tick = 1024, 960
    from audioflow import synth
    rng = np.random.default_rng(6)
    check = sorted({0, S - 1, *rng.choice(np.arange(1, S - 1), 14, replace=False).tolist()})
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    x = np.stack([synth.stream(k, 1.0, 48000) for k in range(S)])
    never, s = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
    for q in (never, s):
        q.enable_wire(gate=True, mem=af.AF_MEM_DEVICE)
        q.enable_wire_features(True, af.AF_MEM_DEVICE)
        q.set_wire_preroll(P)
    gc.collect()                                          # (the counts are the process's: earlier tests' sessions go first)
    held = af.live_allocations()
    s.enable_wire_segments(True, af.AF_MEM_DEVICE)
    grown = af.live_allocations()
    assert grown[0] > held[0]
    lives = {k: SegLife(P, 160) for k in check}
    pieces = 0
    for t in range(45):
        if t == 30:                                       # disabling frees exactly what enabling allocated
            gc.collect()
            before = af.live_allocations()
            s.enable_wire_segments(False)
            after = af.live_allocations()
            assert (before[0] - after[0], before[1] - after[1]) == (grown[0] - held[0], grown[1] - held[1]), (held, grown, before, after)
        xt = x[:, (t % 50) * tick:(t % 50 + 1) * tick]
        l0 = af.kernel_launch_count(); never.push(xt); l1 = af.kernel_launch_count(); rs = s.push(xt)
        l2 = af.kernel_launch_count()
        assert l1 - l0 == l2 - l1, (t, l1 - l0, l2 - l1)
        wn, ws = never.wire(), s.wire()
        pn, bn = _payloads(never, wn)
        ps, bs = _payloads(s, ws)
        for k in range(S):
            assert _strip(wn["streams"][k]) == _strip(ws["streams"][k]) and bn[k] == bs[k]
            assert wn["streams"][k]["n_samples"] == ws["streams"][k]["n_samples"] and np.array_equal(pn[k], ps[k])
        (fn, nn), (fs, ns) = _rows(never), _rows(s)
        assert np.array_equal(nn, ns)
        for k in check:
            assert_bit_equal(fn[k], fs[k])
        if t < 30:
            tab, n = _table(s)
            pieces += int(n.sum())
            for k in check:
                lives[k].tick(orc, tab[k], ws["streams"][k], int(ws["first_frames"][k]), rs["vad"][k])
        else:
            with pytest.raises(ValueError):
                s.wire_segments()
    assert pieces > 100


@pytest.mark.gpu
def test_refusals_leave_the_session_untouched(af, orc):
    """af_session_enable_wire_segments is AF_ERR_INVALID without the wire, ungated, and for a bad mem, and changes
    nothing; af_session_wire_segments refuses before the first push, while the table is off, after an import and after a
    new af_session_enable_wire (which turns the table off)."""
    L = af.load_library()
    S, tick = 4, 960
    xs = np.stack([_bursts(81 + i, 2.0, 48000) for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    ses, twin = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
    rows, st, n = C.c_void_p(), C.c_uint64(), np.zeros(S, np.uint32)
    u32p = C.POINTER(C.c_uint32)

    def query(s):
        return L.af_session_wire_segments(s._h, C.byref(rows), C.byref(st), n.ctypes.data_as(u32p))
    a0 = af.live_allocations()
    assert L.af_session_enable_wire_segments(ses._h, 1, af.AF_MEM_HOST) == af.AF_ERR_INVALID       # the wire is off
    ses.enable_wire(gate=False); twin.enable_wire(gate=False)
    a1 = af.live_allocations()
    assert L.af_session_enable_wire_segments(ses._h, 1, af.AF_MEM_HOST) == af.AF_ERR_INVALID       # not gated
    assert af.live_allocations() == a1 and a1 != a0
    for s in (ses, twin):
        s.enable_wire(gate=True)
        s.enable_wire_features(True)
        s.set_wire_preroll(5)
    a2 = af.live_allocations()
    for bad in (-1, 2, 7):
        assert L.af_session_enable_wire_segments(ses._h, 1, bad) == af.AF_ERR_INVALID
    assert af.live_allocations() == a2
    assert query(ses) == af.AF_ERR_INVALID                                                           # off
    for s in (ses, twin):
        s.enable_wire_segments(True)
    assert query(ses) == af.AF_ERR_INVALID                                                           # no push yet
    for t in range(20):
        x = xs[:, t * tick:(t + 1) * tick]
        ses.push(x); twin.push(x)
        if t == 8:
            assert L.af_session_enable_wire_segments(ses._h, 1, 9) == af.AF_ERR_INVALID
            assert query(ses) == af.AF_OK                                                            # still the last push's
        (a, na), (b, nb) = _table(ses), _table(twin)
        assert np.array_equal(na, nb) and all(p.tobytes() == q.tobytes() for p, q in zip(a, b))
        for g, h in zip(ses.wire()["streams"], twin.wire()["streams"]):
            assert np.array_equal(g["pcm16"], h["pcm16"]) and _strip(g) == _strip(h)
    rec = ses.export_streams([1])
    ses.import_streams([2], rec)
    assert query(ses) == af.AF_ERR_INVALID                                                           # after an import
    ses.push(xs[:, :tick])
    assert query(ses) == af.AF_OK
    ses.enable_wire(gate=True)
    assert ses.segments_mem is None
    ses.push(xs[:, :tick])
    assert query(ses) == af.AF_ERR_INVALID                                                           # enable_wire: off
    assert L.af_session_wire_segments(None, None, None, None) == af.AF_ERR_INVALID
    assert L.af_session_enable_wire_segments(None, 1, af.AF_MEM_HOST) == af.AF_ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
# no GPU
def test_struct_layout_matches_the_header(tmp_path):
    """af_wire_segment: 16 bytes, fields where the header puts them (a C compiler reads the header), and the ctypes and
    numpy mirrors agree; the flag constants too."""
    import audioflow as af
    want = {"frame": 0, "offset": 4, "n_frames": 8, "preroll": 12, "flags": 14, "pad": 15}
    assert C.sizeof(af.WireSegmentC) == 16 and af.WIRE_SEGMENT_DTYPE.itemsize == 16
    for f, o in want.items():
        assert getattr(af.WireSegmentC, f).offset == o and af.WIRE_SEGMENT_DTYPE.fields[f][1] == o, f
    header = open(os.path.join(ROOT, "include", "audioflow_gpu.h")).read()
    assert int(re.search(r"#define\s+AF_WIRE_SEG_CONTINUED\s+(\d+)", header).group(1)) == af.AF_WIRE_SEG_CONTINUED == CONT
    assert int(re.search(r"#define\s+AF_WIRE_SEG_CLOSED\s+(\d+)", header).group(1)) == af.AF_WIRE_SEG_CLOSED == CLOSED
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "l.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "audioflow_gpu.h"\nint main(void){printf("%zu'
                   + "".join(' %zu' for _ in want) + '\\n", sizeof(af_wire_segment)'
                   + "".join(f", offsetof(af_wire_segment, {f})" for f in want) + ');return 0;}\n')
    exe = tmp_path / "l"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [16, *want.values()]


def _no_library():
    raise AssertionError("the library was called")


def test_python_arguments_are_checked_before_the_library(monkeypatch):
    """No GPU: enable_wire_segments refuses a bad mem and a session without the gated wire before it calls the library."""
    import audioflow as af
    monkeypatch.setattr(af, "load_library", _no_library)

    def session(wire_mem=af.AF_MEM_HOST, gate=True):
        s = af.Session.__new__(af.Session)
        s._h, s.S = None, 2
        s.wire_mem, s.wire_gate, s.features_mem, s.wire_preroll, s.segments_mem = wire_mem, gate, None, 0, None
        return s

    for s, mem in ((session(), 2), (session(), -1), (session(), "host"), (session(wire_mem=None), af.AF_MEM_HOST),
                   (session(gate=False), af.AF_MEM_DEVICE)):
        with pytest.raises(ValueError):
            s.enable_wire_segments(True, mem)
    for mem in (af.AF_MEM_HOST, af.AF_MEM_DEVICE):                     # accepted: the call reaches the library
        with pytest.raises(AssertionError):
            session().enable_wire_segments(True, mem)
    with pytest.raises(AssertionError):
        session().enable_wire_segments(False)


def test_new_symbols_in_every_mirror():
    """Both calls are declared in the header, exported by the library and bound by ctypes; the C++ mirror and the Rust
    shim carry them, and the Rust struct has the header's fields in order."""
    import audioflow as af
    header = open(os.path.join(ROOT, "include", "audioflow_gpu.h")).read()
    hpp = open(os.path.join(ROOT, "audio-flow-rs_b200", "host", "audioflow.hpp")).read()
    ffi = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "ffi.rs")).read()
    stream = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "stream.rs")).read()
    L = af.load_library()
    for n in ("af_session_enable_wire_segments", "af_session_wire_segments"):
        assert re.search(r"AF_API\s+int\s+%s\s*\(" % n, header), n
        assert getattr(L, n).restype is C.c_int, n
        assert re.search(r"pub fn %s\s*\(" % n, ffi), n
        assert f"{n}(h_" in hpp and f"ffi::{n}(" in stream, n
    m = re.search(r"pub struct af_wire_segment \{(.*?)\}", ffi, re.S)
    assert m and re.findall(r"pub (\w+):", m.group(1)) == ["frame", "offset", "n_frames", "preroll", "flags", "pad"]
    assert re.search(r"AF_WIRE_SEG_CONTINUED: u8 = 1;", ffi) and re.search(r"AF_WIRE_SEG_CLOSED: u8 = 2;", ffi)
