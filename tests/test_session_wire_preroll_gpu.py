"""Pre-roll of the gated output (af_vad_segments_preroll, af_session_set_wire_preroll): every speech segment reaches back up
to P frames before its detected onset, never into the previous segment and never before the stream's origin.

Batch: af_vad_segments -> af_vad_segments_preroll -> af_vad_gate against orc_vad_segments, the pre-roll rule
(segments_preroll below) and orc_vad_gate.
Sessions, on every tick and stream: n_samples is a whole number of hops (n_frames * hop with features), the base64 is this
tick's PCM16 bytes, the af_wire_tick minus n_samples / n_chars is that of a pre-roll-0 twin session, and the payloads (and
feature rows) concatenated since the stream's origin are orc_vad_gate over the stream's PCM, log-mel and states since its
start, with segments_preroll's segments clamped at the origin."""
import base64
import ctypes as C
import os
import re

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal
from test_session_wire_gpu import _device_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPEECH, ENDING = 1, 2


def _bursts(seed, seconds, rate, ch=1):
    """Tone bursts (80-400 ms) after gaps of 20-500 ms, the first after 40 ms of silence, some with a quiet lead-in: with a
    short silence timeout, segments close and reopen within a pre-roll, and the first onset lies within one of the
    stream's start."""
    rng = np.random.default_rng(seed)
    n = int(seconds * rate)
    x = rng.normal(0.0, 1e-3, n)
    t = np.arange(n) / rate
    pos = int(0.04 * rate)
    while pos < n:
        ln = int(rng.uniform(0.08, 0.4) * rate)
        end = min(n, pos + ln)
        f = rng.uniform(150.0, 3000.0)
        env = np.full(end - pos, rng.choice([0.05, 0.2, 0.5]))
        lead = min(end - pos, int(rng.uniform(0.0, 0.06) * rate))
        env[:lead] *= np.linspace(0.02, 1.0, lead)                # a quiet lead-in below the threshold
        x[pos:end] += env * np.sin(2 * np.pi * f * t[pos:end])
        pos = end + int(rng.choice([rng.uniform(0.02, 0.12), rng.uniform(0.12, 0.5)]) * rate)
    x = np.clip(x, -1.0, 1.0).astype(np.float32)
    return np.repeat(x, ch) if ch > 1 else x


def segments_preroll(seg, P, n_seg=None):
    """The pre-roll rule on a segment list ([n, 2] frames, [start, end)): each of the first min(n_seg, n) segments starts
    at max(start - P, end of the previous segment, 0), the first one's predecessor ending at 0; ends are kept."""
    out = np.array(seg, np.int64).reshape(-1, 2)
    for k in range(min(len(out) if n_seg is None else n_seg, len(out))):
        lo = out[k - 1, 1] if k else 0
        out[k, 0] = max(out[k, 0] - P, lo, 0)
    return out.astype(np.uint32)


def _vad(af, **kw):
    return af.VadConfig(**{"silence_timeout_frames": 2, "min_speech_frames": 1, **kw})


def _rows(ses):
    """The wire features of the last push as per-stream [n, n_mels] arrays (device rows copied to the host)."""
    import audioflow as af
    rows, n = ses.wire_features()
    if ses.features_mem == af.AF_MEM_DEVICE:
        ptr, stride = rows
        M = ses.pipe.cfg.n_mels
        allr = _device_rows(ptr, ses.S, stride, np.float32)
        rows = [allr[k, :int(n[k]) * M].reshape(-1, M).copy() for k in range(ses.S)]
    return rows, n


def _payloads(ses, w):
    """Per-stream PCM16 payloads and base64 texts of the last push (device rows copied to the host)."""
    import audioflow as af
    st = w["streams"]
    if ses.wire_mem == af.AF_MEM_HOST:
        return [g["pcm16"] for g in st], [g["base64"] for g in st]
    p = _device_rows(w["pcm16_ptr"], ses.S, w["pcm16_stride"], np.int16)
    b = _device_rows(w["base64_ptr"], ses.S, w["base64_stride"], np.uint8)
    return ([p[k, :g["n_samples"]].copy() for k, g in enumerate(st)],
            [b[k, :g["n_chars"]].tobytes() for k, g in enumerate(st)])


def _strip(g):
    return {q: v for q, v in g.items() if q not in ("pcm16", "base64", "n_samples", "n_chars")}


class _Life:
    """One stream since its start: everything the session emitted for it, and its payloads since its origin."""

    def __init__(self):
        self.pcm, self.lm, self.vad, self.pay, self.feat = [], [], [], [], []
        self.origin = 0

    def frames(self):
        return sum(len(v) for v in self.vad)

    def new_origin(self):
        self.origin, self.pay, self.feat = self.frames(), [], []


def check_life(orc, L, P, hop, M):
    """Stream L's payloads since its origin == orc_vad_gate over its life with the pre-rolled segments clamped there."""
    st = np.concatenate(L.vad) if L.vad else np.zeros(0, np.uint8)
    segs = orc.vad_segments(st)
    ext = segments_preroll(segs, P)
    clamped = np.array([[max(int(a), L.origin), int(b)] for a, b in ext if b > L.origin], np.uint32).reshape(-1, 2)
    pcm = np.concatenate(L.pcm) if L.pcm else np.zeros(0, np.float32)
    lm = np.concatenate(L.lm).reshape(-1, M) if M else None
    gp, gl, _ = orc.vad_gate(pcm, lm, clamped, hop)
    got = np.concatenate(L.pay) if L.pay else np.zeros(0, np.int16)
    assert np.array_equal(got, orc.pcm16_encode(gp)), (len(got), len(gp), L.origin, clamped[:4])
    if M:
        assert_bit_equal(np.concatenate(L.feat).reshape(-1, M) if L.feat else np.zeros((0, M), np.float32), gl, "feature rows")
    return len(clamped)


class Driver:
    """A session of `formats` with the gated wire (and, with fmem, its features) and pre-roll P, pushed ticks from
    per-stream sources, beside a pre-roll-0 twin session fed the same ticks; streams in `twins` also have one-stream twins
    with the same pre-roll.  Every tick checks every stream (see check_life)."""

    def __init__(self, af, orc, pipe, formats, stream_format, P, fmem=None, wmem=None, twins=(), seconds=8.0, hop=160,
                 check=None):
        self.af, self.orc, self.pipe, self.formats, self.P, self.hop = af, orc, pipe, formats, P, hop
        self.M = pipe.cfg.n_mels if fmem is not None else 0
        wmem = af.AF_MEM_HOST if wmem is None else wmem

        def make(sf):
            s = af.Session.formats(pipe, formats, sf)
            s.enable_wire(gate=True, mem=wmem)
            if fmem is not None:
                s.enable_wire_features(True, fmem)
            return s
        self.ses, self.zero = make(stream_format), make(stream_format)
        self.ses.set_wire_preroll(P)
        self.S = self.ses.S
        self.check = range(self.S) if check is None else check
        self.src = [_bursts(300 + 11 * k, seconds, *formats[f][:2]) for k, f in enumerate(stream_format)]
        self.cur = [0] * self.S
        self.life = [_Life() for _ in range(self.S)]
        self.twin = {}
        for k in twins:
            self.twin[k] = make([int(stream_format[k])])
            self.twin[k].set_wire_preroll(P)
        self.grown = 0                                               # ticks whose payload the pre-roll made longer
        self.n_seg = 0

    def samples(self, k, frames):
        ch = self.formats[self.ses.stream_format[k]][1]
        n = frames * ch
        if self.cur[k] + n > len(self.src[k]):
            self.cur[k] = 0
        x = self.src[k][self.cur[k]:self.cur[k] + n]
        self.cur[k] += n
        return x

    def tick(self, frames, end=None, lockstep=False):
        end = [False] * self.S if end is None else [bool(e) for e in end]
        xs = [self.samples(k, n) for k, n in enumerate(frames)]
        push = (lambda s: s.push(np.stack(xs))) if lockstep else (lambda s: s.push_streams(xs, end))
        l0 = self.af.kernel_launch_count()
        push(self.zero)
        l1 = self.af.kernel_launch_count()
        r = push(self.ses)
        self.launches = (l1 - l0, self.af.kernel_launch_count() - l1)
        w, wz = self.ses.wire(), self.zero.wire()
        pays, texts = _payloads(self.ses, w)
        rows, nf = _rows(self.ses) if self.M else (None, None)
        for k in range(self.S):
            g, gz = w["streams"][k], wz["streams"][k]
            assert _strip(g) == _strip(gz), (k, g, gz)
            assert g["n_samples"] % self.hop == 0 and g["n_samples"] >= gz["n_samples"], (k, g["n_samples"], gz["n_samples"])
            self.grown += g["n_samples"] > gz["n_samples"]
            if k not in self.check:
                continue
            assert len(pays[k]) == g["n_samples"]
            assert texts[k] == base64.b64encode(pays[k].astype("<i2").tobytes()) and g["n_chars"] == len(texts[k]), k
            if self.M:
                assert int(nf[k]) * self.hop == g["n_samples"], (k, int(nf[k]), g["n_samples"])
            L = self.life[k]
            L.pcm.append(np.asarray(r["pcm"][k])); L.vad.append(np.asarray(r["vad"][k]))
            if self.M:
                L.lm.append(np.asarray(r["logmel"][k]).reshape(-1, self.M)); L.feat.append(rows[k])
            L.pay.append(pays[k])
            self.n_seg = max(self.n_seg, check_life(self.orc, L, self.P, self.hop, self.M))
        for k, t in self.twin.items():
            t.push_streams([xs[k]], [end[k]])
            tw = t.wire()
            tp, _ = _payloads(t, tw)
            assert tw["streams"][0]["n_samples"] == w["streams"][k]["n_samples"], k
            assert np.array_equal(tp[0], pays[k]), f"stream {k} payload vs its twin"
            if self.M:
                tr, _ = _rows(t)
                assert_bit_equal(tr[0], rows[k], f"stream {k} rows vs its twin")
        for k in range(self.S):
            if end[k]:
                self.life[k] = _Life()
        return r

    def reset(self, ids):
        self.ses.reset_streams(ids); self.zero.reset_streams(ids)
        for k in ids:
            if k in self.twin:
                self.twin[k].reset_streams([0])
            self.life[k] = _Life()

    def restart(self, ids, fmts):
        self.ses.restart_streams(ids, fmts); self.zero.restart_streams(ids, fmts)
        for k, f in zip(ids, fmts):
            if k in self.twin:
                self.twin[k].restart_streams([0], [f])
            self.life[k] = _Life()
            self.src[k] = _bursts(900 + k, 8.0, *self.formats[f][:2])
            self.cur[k] = 0

    def set_vad_configs(self, ids, cfgs):
        for s in (self.ses, self.zero):
            s.set_vad_configs(ids, cfgs)
        for k, c in zip(ids, cfgs):
            if k in self.twin:
                self.twin[k].set_vad_configs([0], [c])

    def set_preroll(self, P):
        self.ses.set_wire_preroll(P)
        for t in self.twin.values():
            t.set_wire_preroll(P)
        self.P = P
        for L in self.life:
            L.new_origin()


# ---------------------------------------------------------------------------------------------------------------------
# batch
@pytest.mark.gpu
@pytest.mark.parametrize("P", [0, 1, 3, 30, 100, 10 ** 6])
def test_batch_segments_preroll_gate(af, orc, P):
    """A ragged batch (mixed rates and lengths, an empty stream, one without speech; segment capacities 64 and 2):
    af_vad_segments -> af_vad_segments_preroll -> af_vad_gate is bit for bit orc_vad_segments -> segments_preroll -> orc_vad_gate in
    PCM, log-mel rows and offsets.  P = 0 leaves the segments byte-identical."""
    import torch
    dev = torch.device("cuda")
    L = af.load_library()
    M = 80
    specs = [(210, 6.0, 48000), (211, 4.1, 44100), (212, 0.0, 48000), (213, 3.3, 16000), (214, 9.7, 48000)]
    streams = [(_bursts(i, sec, rate), rate) for (i, sec, rate) in specs]
    streams.append((np.full(48000 * 2, 1e-4, np.float32), 48000))
    S = len(streams)
    arrs = [torch.tensor(x, device=dev) if len(x) else torch.zeros(4, device=dev) for x, _ in streams]
    pipe = af.Pipeline(af.pipeline_config(n_mels=M, vad=_vad(af)))
    b = pipe.batch([(a.data_ptr(), len(x), r, 1, af.AF_FMT_F32) for a, (x, r) in zip(arrs, streams)], af.AF_MEM_DEVICE)
    pcm = torch.zeros((S, b.pcm_stride), device=dev); lm = torch.zeros((S, b.logmel_stride), device=dev)
    vad = torch.zeros((S, b.vad_stride), device=dev, dtype=torch.uint8)
    torch.cuda.synchronize()
    b.run_device(b.outputs_struct(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, vad.data_ptr(), b.vad_stride))
    checked = 0
    for seg_cap in (64, 2):
        seg = torch.zeros((S, seg_cap, 2), device=dev, dtype=torch.int32)
        nseg = torch.zeros(S, device=dev, dtype=torch.int32)
        nfr = torch.tensor(b.n_vad[:S].astype(np.int32), device=dev)
        nout = torch.tensor(b.n_out[:S].astype(np.int32), device=dev)
        torch.cuda.synchronize()
        assert L.af_vad_segments(vad.data_ptr(), b.vad_stride, nfr.data_ptr(), S, seg.data_ptr(), seg_cap, nseg.data_ptr(), None) == 0
        before = seg.cpu().numpy().copy()
        assert L.af_vad_segments_preroll(seg.data_ptr(), seg_cap, nseg.data_ptr(), S, P, None) == 0
        after = seg.cpu().numpy()
        if P == 0:
            assert before.tobytes() == after.tobytes()
        g_pcm = torch.full((S, b.pcm_stride), float("nan"), device=dev)       # (pre-roll stays within the stream)
        g_lm = torch.full((S, b.logmel_stride), float("nan"), device=dev)
        g_off = torch.zeros((S, seg_cap + 1), device=dev, dtype=torch.int32)
        g_n = torch.zeros(S, device=dev, dtype=torch.int32)
        go = af.GateOutputsC(g_pcm.data_ptr(), g_pcm.shape[1], g_lm.data_ptr(), g_lm.shape[1], g_off.data_ptr(), g_n.data_ptr())
        torch.cuda.synchronize()
        af._check(L.af_vad_gate(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, M, nout.data_ptr(), 160,
                                seg.data_ptr(), seg_cap, nseg.data_ptr(), S, C.byref(go), None))
        torch.cuda.synchronize()
        for i in range(S):
            T, n_out = int(b.n_vad[i]), int(b.n_out[i])
            full = orc.vad_segments(vad[i, :T].cpu().numpy())
            exp = segments_preroll(full[:seg_cap], P, len(full))
            n = min(int(nseg[i]), seg_cap)
            assert n == len(exp)
            assert np.array_equal(after[i, :n].astype(np.uint32), exp), (i, after[i, :n], exp)
            assert (after[i, n:] == before[i, n:]).all()                  # slots past the segments are not touched
            rp, rl, roff = orc.vad_gate(pcm[i, :n_out].cpu().numpy(), lm[i, :T * M].reshape(T, M).cpu().numpy(), exp, 160)
            kept = int(roff[-1])
            assert int(g_n[i]) == kept
            assert np.array_equal(g_off[i, :n + 1].cpu().numpy().astype(np.uint32), roff)
            assert_bit_equal(g_pcm[i, :kept * 160].cpu().numpy(), rp, f"gated pcm {i}")
            assert_bit_equal(g_lm[i, :kept * M].cpu().numpy(), rl.reshape(-1), f"gated log-mel {i}")
            checked += len(exp)
    assert checked > 10


# ---------------------------------------------------------------------------------------------------------------------
# sessions
@pytest.mark.gpu
@pytest.mark.parametrize("fmem,wmem", [("host", "host"), ("device", "device"), (None, "host")])
def test_20ms_ticks_history_spans_many_pushes(af, orc, fmem, wmem):
    """Lockstep 20 ms ticks at 48 kHz and P = 30 (15 ticks of history), with and without features, host and device rows:
    segments close and reopen within P frames, and the first onsets lie within P frames of the origin."""
    H, D = af.AF_MEM_HOST, af.AF_MEM_DEVICE
    fm = None if fmem is None else (H if fmem == "host" else D)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = Driver(af, orc, pipe, [(48000, 1, 960)], [0] * 5, 30, fm, H if wmem == "host" else D)
    for t in range(300):
        d.tick([960] * d.S, lockstep=True)
    assert d.grown > 20 and d.n_seg >= 3
    st = np.concatenate(d.life[0].vad)
    segs = orc.vad_segments(st)
    assert segs[0, 0] < 30 and (segs[1:, 0] - segs[:-1, 1] < 30).any()   # the cases the pre-roll is clamped in


@pytest.mark.gpu
@pytest.mark.parametrize("P", [3, 30])
def test_1s_ticks_several_segments_per_tick(af, orc, P):
    """1 s ticks: several segments start in one tick, each with its own pre-roll out of the same tick."""
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = Driver(af, orc, pipe, [(48000, 1, 48000), (44100, 2, 88200)], [0, 1, 0, 1], P, af.AF_MEM_HOST, twins=(1,))
    most = 0
    for t in range(7):
        d.tick([d.formats[f][2] // d.formats[f][1] for f in d.ses.stream_format])
        most = max(most, max(g["started"] for g in d.ses.wire()["streams"]))
    assert most >= 2 and d.grown > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mem", ["host", "device"])
def test_ragged_mixed_formats_ends_resets_restarts(af, orc, mem):
    """12 streams in four capture formats, ragged ticks, ends, reset_streams, restart_streams into another format,
    per-stream VAD configurations set and changed mid-stream; six streams have one-stream twins with the same pre-roll."""
    m = af.AF_MEM_HOST if mem == "host" else af.AF_MEM_DEVICE
    rng = np.random.default_rng(11 + m)
    formats = [(48000, 1, 960), (44100, 1, 882), (16000, 1, 320), (48000, 2, 1920)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = Driver(af, orc, pipe, formats, [k % 4 for k in range(12)], 12, m, m, twins=(0, 1, 2, 3, 6, 11))
    V = af.VadConfig
    d.set_vad_configs([1, 2, 6], [V(threshold_db=-40.0, min_speech_frames=1), V(smoothing_factor=0.6, silence_timeout_frames=4),
                                  V(threshold_db=-55.0, silence_timeout_frames=2)])
    for t in range(90):
        counts = []
        for k in range(d.S):
            mx = formats[d.ses.stream_format[k]][2] // formats[d.ses.stream_format[k]][1]
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
    assert d.grown > 10


@pytest.mark.gpu
def test_preroll_set_and_changed_mid_stream(af, orc):
    """The pre-roll set at push 20, changed to 40 at 60, to 0 at 100 and to 7 at 120: every call makes the next push
    every stream's origin; a twin session that makes the same calls at the same pushes computes the same payloads."""
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = Driver(af, orc, pipe, [(48000, 1, 960)], [0] * 4, 0, af.AF_MEM_DEVICE, twins=(0, 3))
    for t in range(160):
        if t in (20, 60, 100, 120):
            d.set_preroll({20: 10, 60: 40, 100: 0, 120: 7}[t])
        d.tick([960] * d.S, lockstep=True)
    assert d.grown > 10


@pytest.mark.gpu
def test_vad_20ms_frames_pcm_only(af, orc):
    """VAD on 20 ms frames (vad_frame_len = vad_hop = 320), no log-mel: pre-roll in hops of 320 samples."""
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad=_vad(af), vad_frame_len=320, vad_hop=320))
    d = Driver(af, orc, pipe, [(48000, 1, 1920), (16000, 1, 640)], [0, 1, 0, 1], 9, None, hop=320, twins=(1,))
    rng = np.random.default_rng(3)
    for t in range(120):
        d.tick([int(rng.integers(0, d.formats[f][2] + 1)) for f in d.ses.stream_format])
    assert d.grown > 5


@pytest.mark.gpu
@pytest.mark.parametrize("dst_mem", ["host", "device"])
def test_import_is_an_origin(af, orc, dst_mem):
    """A stream exported mid-utterance from session A and imported into session B (pre-roll on): from the import on, its
    payloads are orc_vad_gate over its life with the origin at the import; record_bytes() does not depend on the
    pre-roll; one launch clears the history of every imported slot."""
    m = af.AF_MEM_HOST if dst_mem == "host" else af.AF_MEM_DEVICE
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    rate, tick, P = 44100, 882, 25
    x = _bursts(77, 6.0, rate)
    a = af.Session(pipe, 4, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session.formats(pipe, [(16000, 1, 320), (rate, 1, 2 * tick)], [0] * 6)
    rb0 = b.record_bytes()
    for s in (a, b):
        s.enable_wire(gate=True, mem=m)
        s.enable_wire_features(True, m)
        s.set_wire_preroll(P)
    assert b.record_bytes() == rb0 == a.record_bytes()
    slot_a, slot_b = 2, 4
    empty = np.zeros(0, np.float32)
    L = _Life()
    moved = False
    for t in range(250):
        chunk = x[t * tick:(t + 1) * tick]
        ses, slot = (b, slot_b) if moved else (a, slot_a)
        if not moved:
            b.push_streams([empty] * b.S)
        r = ses.push_streams([chunk if k == slot else empty for k in range(ses.S)])
        pays, _ = _payloads(ses, ses.wire())
        rows, _ = _rows(ses)
        L.pcm.append(r["pcm"][slot]); L.vad.append(r["vad"][slot]); L.lm.append(r["logmel"][slot]); L.pay.append(pays[slot])
        L.feat.append(rows[slot])
        check_life(orc, L, P, 160, 80)
        if t == 120:
            rec = a.export_streams([slot_a])
            assert rec.shape[1] == rb0
            l0 = af.kernel_launch_count()
            b.import_streams([slot_b], rec)
            assert af.kernel_launch_count() - l0 == 2                # unpack, history clear
            a.reset_streams([slot_a])
            L.new_origin()
            moved = True
    assert len(np.concatenate(L.pay)) > 0


@pytest.mark.gpu
def test_1024_streams_and_launches(af, orc):
    """cfg5's shape (1024 x 20 ms at 48 kHz, 80 mels, VAD, gated wire with features): a tick with the pre-roll launches
    one kernel fewer than one without (it replaces the features and wire kernels); 16 streams checked per tick."""
    S, tick, n_ticks = 1024, 960, 40
    rng = np.random.default_rng(5)
    check = sorted({0, S - 1, *rng.choice(np.arange(1, S - 1), 14, replace=False).tolist()})
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    d = Driver(af, orc, pipe, [(48000, 1, tick)], [0] * S, 30, af.AF_MEM_DEVICE, af.AF_MEM_DEVICE, seconds=1.0, check=check)
    for t in range(n_ticks):
        d.tick([tick] * S, lockstep=True)
        if t > 0:                                 # ingest+resample, fused (2), scan, features + wire / pre-roll
            assert d.launches == (6, 5), d.launches
    assert d.grown > 50


@pytest.mark.gpu
def test_back_to_zero_is_never_set(af, orc):
    """A session whose pre-roll went to 30 and back to 0 computes, with the same launches, the payloads and feature rows of
    one that never set one; its allocations return to where they were."""
    S, tick = 6, 960
    xs = np.stack([_bursts(40 + i, 3.0, 48000) for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    never, back = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
    for s in (never, back):
        s.enable_wire(gate=True)
        s.enable_wire_features(True, af.AF_MEM_HOST)
        s.push(xs[:, :tick]); s.push(xs[:, tick:2 * tick])
    held = af.live_allocations()
    back.set_wire_preroll(30)
    assert af.live_allocations()[0] > held[0]
    for t in range(2, 40):
        never.push(xs[:, t * tick:(t + 1) * tick]); back.push(xs[:, t * tick:(t + 1) * tick])
    back.set_wire_preroll(0)
    assert af.live_allocations() == held
    with pytest.raises(ValueError):
        back.wire()                                               # the rows were replaced
    for t in range(40, 90):
        x = xs[:, t * tick:(t + 1) * tick]
        l0 = af.kernel_launch_count(); never.push(x); l1 = af.kernel_launch_count(); back.push(x); l2 = af.kernel_launch_count()
        assert l1 - l0 == l2 - l1
        wn, wb = never.wire(), back.wire()
        for g, h in zip(wn["streams"], wb["streams"]):
            assert g["base64"] == h["base64"] and np.array_equal(g["pcm16"], h["pcm16"]) and _strip(g) == _strip(h)
        (rn, nn), (rb, nb) = _rows(never), _rows(back)
        assert np.array_equal(nn, nb)
        for k in range(S):
            assert_bit_equal(rn[k], rb[k], f"tick {t} stream {k}")


@pytest.mark.gpu
def test_enable_calls_set_the_preroll_back(af, orc):
    """enable_wire_features (on or off) and enable_wire set the pre-roll back to 0: the payloads are then those of a
    session that never set one."""
    S, tick = 3, 960
    xs = np.stack([_bursts(60 + i, 2.0, 48000) for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    for call in ("features_on", "features_off", "wire"):
        never, s = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
        for q in (never, s):
            q.enable_wire(gate=True)
        s.set_wire_preroll(20)
        for t in range(30):
            never.push(xs[:, t * tick:(t + 1) * tick]); s.push(xs[:, t * tick:(t + 1) * tick])
        if call == "features_on":
            s.enable_wire_features(True); never.enable_wire_features(True)
        elif call == "features_off":
            s.enable_wire_features(False)
        else:
            s.enable_wire(gate=True)
        assert s.wire_preroll == 0
        for t in range(30, 60):
            x = xs[:, t * tick:(t + 1) * tick]
            never.push(x); s.push(x)
            for g, h in zip(never.wire()["streams"], s.wire()["streams"]):
                assert np.array_equal(g["pcm16"], h["pcm16"]) and _strip(g) == _strip(h), call


@pytest.mark.gpu
def test_refusals_leave_the_session_untouched(af, orc):
    """set_wire_preroll is AF_ERR_INVALID without the gated wire and above AF_WIRE_PREROLL_MAX, and changes nothing: the
    session then computes what a twin that never met the refusals computes."""
    L = af.load_library()
    S, tick = 4, 960
    xs = np.stack([_bursts(80 + i, 2.0, 48000) for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80, vad=_vad(af)))
    ses, twin = (af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick) for _ in range(2))
    assert L.af_session_set_wire_preroll(ses._h, 5) == af.AF_ERR_INVALID          # the wire is off
    ses.enable_wire(gate=False)
    assert L.af_session_set_wire_preroll(ses._h, 5) == af.AF_ERR_INVALID          # not gated
    for s in (ses, twin):
        s.enable_wire(gate=True)
        s.enable_wire_features(True, af.AF_MEM_DEVICE)
        s.set_wire_preroll(12)
    for t in range(40):
        x = xs[:, t * tick:(t + 1) * tick]
        ses.push(x); twin.push(x)
        if t in (10, 20):
            a0 = af.live_allocations()
            assert L.af_session_set_wire_preroll(ses._h, af.AF_WIRE_PREROLL_MAX + 1) == af.AF_ERR_INVALID
            assert L.af_session_set_wire_preroll(ses._h, 0xffffffff) == af.AF_ERR_INVALID
            assert af.live_allocations() == a0
            ses.wire()                                            # the rows of the last push are still valid
        for g, h in zip(ses.wire()["streams"], twin.wire()["streams"]):
            assert np.array_equal(g["pcm16"], h["pcm16"]) and g["base64"] == h["base64"] and _strip(g) == _strip(h)
            assert g["n_samples"] == h["n_samples"]
        (r1, n1), (r2, n2) = _rows(ses), _rows(twin)
        assert np.array_equal(n1, n2)
        for k in range(S):
            assert_bit_equal(r1[k], r2[k])
    assert L.af_session_set_wire_preroll(None, 1) == af.AF_ERR_INVALID
    assert L.af_vad_segments_preroll(None, 4, None, 1, 3, None) == af.AF_ERR_INVALID


# ---------------------------------------------------------------------------------------------------------------------
# no GPU
def _frames_by_definition(states, P):
    """The frames the pre-roll keeps, restated frame by frame: a kept frame (Speech, or Ending right after Speech), or a
    frame at most P before a segment start (Speech after a frame that is not) with no kept frame in between."""
    st = np.asarray(states, np.uint8)
    pre = np.concatenate([[0], st[:-1]]).astype(np.uint8)
    kept = (st == SPEECH) | ((st == ENDING) & (pre == SPEECH))
    start = (st == SPEECH) & (pre != SPEECH)
    keep = kept.copy()
    for g in np.nonzero(start)[0]:
        f = g - 1
        while f >= 0 and f >= g - P and not kept[f]:
            keep[f] = True
            f -= 1
    return np.nonzero(keep)[0]


def test_preroll_rule_against_its_definition(orc):
    """segments_preroll on orc_vad_segments' segments covers exactly the frames of the frame-by-frame definition, on random
    state sequences with gaps shorter than P, onsets before frame P and P beyond the stream's length; with fewer slots than
    segments, only the listed segments move."""
    rng = np.random.default_rng(1)
    seen = dict(short_gap=0, early=0, overflow=0)
    for trial in range(400):
        T = int(rng.integers(0, 400))
        st = np.zeros(T, np.uint8)
        f = int(rng.integers(0, 12))
        while f < T:
            n = int(rng.integers(1, 25))
            st[f:f + n] = SPEECH
            if f + n < T and rng.random() < 0.6:
                st[f + n] = ENDING
            f += n + 1 + int(rng.integers(0, 40))
        segs = orc.vad_segments(st)
        P = int(rng.choice([0, 1, 3, 7, 30, 100, 1000, 10 ** 6]))
        got = segments_preroll(segs, P)
        frames = np.concatenate([np.arange(a, b) for a, b in got]) if len(got) else np.zeros(0, np.int64)
        assert np.array_equal(frames, _frames_by_definition(st, P)), (trial, P)
        assert np.array_equal(got[:, 1], segs[:, 1])
        cap = int(rng.integers(0, len(segs) + 1))
        part = segments_preroll(segs[:cap], P, len(segs))
        assert np.array_equal(part, got[:cap])
        seen["short_gap"] += bool(len(segs) > 1 and (segs[1:, 0] - segs[:-1, 1] < P).any())
        seen["early"] += bool(len(segs) and segs[0, 0] < P)
        seen["overflow"] += cap < len(segs)
    assert min(seen.values()) > 10, seen


def _no_library():
    raise AssertionError("the library was called")


def test_python_arguments_are_checked_before_the_library(monkeypatch):
    """No GPU: set_wire_preroll refuses a count out of range or not an integer, and a session without the gated wire,
    before it calls the library."""
    import audioflow as af
    monkeypatch.setattr(af, "load_library", _no_library)

    def session(wire_mem=af.AF_MEM_HOST, gate=True):
        s = af.Session.__new__(af.Session)
        s._h, s.S = None, 2
        s.wire_mem, s.wire_gate, s.features_mem, s.wire_preroll = wire_mem, gate, None, 0
        return s

    for s, P in ((session(), -1), (session(), af.AF_WIRE_PREROLL_MAX + 1), (session(), 2.5), (session(), True),
                 (session(), "3"), (session(wire_mem=None), 3), (session(gate=False), 3)):
        with pytest.raises(ValueError):
            s.set_wire_preroll(P)
    for P in (0, 1, af.AF_WIRE_PREROLL_MAX, np.uint32(7)):              # accepted: the call reaches the library
        with pytest.raises(AssertionError):
            session().set_wire_preroll(P)


def test_new_symbols_in_every_mirror():
    """Both calls and AF_WIRE_PREROLL_MAX are declared in the header, exported by the library and bound by ctypes; the
    C++ mirror and the Rust shim carry them."""
    import audioflow as af
    header = open(os.path.join(ROOT, "include", "audioflow_gpu.h")).read()
    hpp = open(os.path.join(ROOT, "audio-flow-rs_b200", "host", "audioflow.hpp")).read()
    ffi = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "ffi.rs")).read()
    stream = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "stream.rs")).read()
    L = af.load_library()
    for n in ("af_vad_segments_preroll", "af_session_set_wire_preroll"):
        assert re.search(r"AF_API\s+int\s+%s\s*\(" % n, header), n
        assert getattr(L, n).restype is C.c_int, n
        assert re.search(r"pub fn %s\s*\(" % n, ffi), n
    assert "af_session_set_wire_preroll(" in hpp and "ffi::af_session_set_wire_preroll(" in stream
    m = re.search(r"#define\s+AF_WIRE_PREROLL_MAX\s+(\d+)", header)
    assert m and int(m.group(1)) == af.AF_WIRE_PREROLL_MAX
    assert re.search(r"AF_WIRE_PREROLL_MAX: u32 = %d;" % af.AF_WIRE_PREROLL_MAX, ffi)
