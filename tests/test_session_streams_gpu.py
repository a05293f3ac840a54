"""Sessions whose streams have their own timelines (af_session_push_streams, af_session_reset_streams,
af_session_push_rings_available, af_session_wire_first_frames).  Stream k of a session must behave exactly like a one-stream
session pushed the same ticks: per tick BatchResampler::process (resampler.rs:132-147) on the stream's own samples, flush
(resampler.rs:150-166) on an end, the VAD over the frames completed, the wire payload and record of those frames, its levels;
and start afresh after an end or a reset.  Everything is checked against the oracle objects: PCM, VAD states, detector
states (smoothed energy included) and wire payloads bit-exact, log-mel within assert_logmel_close."""
import ctypes as C

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal, assert_logmel_close
from test_session_wire_gpu import _b64, _bursts, _device_rows, _oracle_events

SPEECH = 1


def _source(orc, seed, seconds, rate, ch, fmt):
    """A long interleaved signal a stream reads its ticks from (bursts of tone: segments open and close often)."""
    x = _bursts(seed, seconds, rate)
    if ch > 1:
        x = np.repeat(x, ch) * np.tile(np.linspace(1.0, 0.5, ch, dtype=np.float32), len(x))
    if fmt == "i16":
        return np.round(np.clip(x, -1, 1) * 32767).astype(np.int16)
    return x.astype(np.float32)


class _Life:
    """One stream from a start to its end / reset, as the reference objects see it."""

    def __init__(self, orc, rate):
        self.b = orc.BatchResampler(rate, 16000)
        self.pcm, self.lm, self.vad, self.frames, self.payload, self.records = [], [], [], [], [], []
        self.det, self.carry = orc.VoiceActivityDetector(), np.zeros(0, np.float32)


class Harness:
    """Drives a session with ragged ticks and checks every stream in `check` against its own reference objects."""

    def __init__(self, af, orc, S, rate, ch=1, fmt="f32", max_tick=960, n_mels=80, vad_len=0, vad_hop=0, check=None,
                 wire=None, levels=False, seconds=30.0):
        self.af, self.orc, self.S, self.rate, self.ch, self.fmt = af, orc, S, rate, ch, fmt
        self.n_mels, self.flen, self.hop = n_mels, vad_len or 400, vad_hop or 160
        self.pipe = af.Pipeline(af.pipeline_config(n_mels=n_mels, vad_frame_len=vad_len, vad_hop=vad_hop))
        self.ses = af.Session(self.pipe, S, rate, ch, af.AF_FMT_I16 if fmt == "i16" else af.AF_FMT_F32, max_tick_samples=max_tick)
        self.check = set(range(S)) if check is None else set(check)
        base = [_source(orc, 300 + i, seconds, rate, ch, fmt) for i in range(4)]
        self.src = [np.roll(base[k % 4], -ch * ((k * 1237) % 20000)) if k in self.check else base[k % 4] for k in range(S)]
        self.cur = [0] * S
        self.life = {k: _Life(orc, rate) for k in self.check}
        self.wire, self.levels = wire, levels
        if wire is not None:
            self.ses.enable_wire(gate=wire[0], mem=wire[1])
        if levels:
            self.ses.enable_levels()
        self.closed, self.just_ended = 0, set()

    def samples(self, counts):
        xs = []
        for k, n in enumerate(counts):
            if self.cur[k] + n > len(self.src[k]):
                self.cur[k] = 0
            xs.append(self.src[k][self.cur[k]:self.cur[k] + n])
            self.cur[k] += n
        return xs

    def _mono(self, x):
        xi = self.orc.i16_to_f32(x) if self.fmt == "i16" else np.asarray(x, np.float32)
        return self.orc.to_mono(xi, self.ch)

    def tick(self, counts, end=None, xs=None, result=None):
        """Push one tick (or check `result` of a tick already pushed with samples xs) and compare every checked stream."""
        if xs is None:
            xs = self.samples(counts)
        r = result if result is not None else self.ses.push_streams(xs, end)
        w = self.ses.wire() if self.wire is not None else None
        lv = self.ses.levels() if self.levels else None
        self.just_ended = set()
        for k in sorted(self.check):
            L = self.life[k]
            fin = end is not None and bool(end[k])
            y = L.b.process(self._mono(xs[k]))
            if fin:
                y = np.concatenate([y, L.b.flush()])
            assert int(r["n_pcm"][k]) == len(y), (k, int(r["n_pcm"][k]), len(y))
            assert_bit_equal(r["pcm"][k], y, f"stream {k} pcm")
            before = self.orc.num_frames(sum(len(p) for p in L.pcm), self.flen, self.hop)
            L.pcm.append(y)
            T = self.orc.num_frames(sum(len(p) for p in L.pcm), self.flen, self.hop) - before
            assert int(r["n_vad"][k]) == T, (k, int(r["n_vad"][k]), T)
            L.frames.append(T)
            L.vad.append(r["vad"][k])
            if self.n_mels:
                L.lm.append(r["logmel"][k])
            if w is not None:
                self._wire_tick(k, L, w, y, before)
            if lv is not None:
                self._levels_tick(k, L, lv, y)
            if fin:
                self.close(k, r["vad_final"][k], ended=True)
                self.just_ended.add(k)
        return r

    def _wire_tick(self, k, L, w, y, before):
        g = w["streams"][k]
        assert int(w["first_frames"][k]) == before, (k, int(w["first_frames"][k]), before)
        if k == 0:
            assert w["first_frame"] == before
        if self.wire[1] == self.af.AF_MEM_HOST:
            pcm16 = g["pcm16"]
            assert g["base64"] == _b64(pcm16)
        else:
            n = g["n_samples"]
            rows = _device_rows(w["pcm16_ptr"], self.S, w["pcm16_stride"], np.int16)
            pcm16 = rows[k, :n]
            b = _device_rows(w["base64_ptr"], self.S, w["base64_stride"], np.uint8)[k, :g["n_chars"]].tobytes()
            assert b == _b64(pcm16)
        if not self.wire[0]:
            assert_bit_equal(pcm16, self.orc.pcm16_encode(y), f"stream {k} ungated payload")
            assert g["base64"] is None or g["base64"] == self.orc.pcm16_base64(y)
        L.payload.append(np.asarray(pcm16, np.int16))
        L.records.append((before, g["started"], g["ended"], g["in_speech"], g["continued"], g["n_samples"]))

    def _levels_tick(self, k, L, lv, y):
        want_peak = np.float32(np.max(np.abs(y))) if len(y) else np.float32(0)
        assert lv["peak"][k].view(np.uint32) == want_peak.view(np.uint32), k
        L.carry = np.concatenate([L.carry, y])
        while len(L.carry) >= 400:
            L.det.detect(L.carry[:400])
            L.carry = L.carry[160:]
        want_db, got_db = np.float32(L.det.energy_db()), lv["level_db"][k]
        assert (np.isneginf(want_db) and np.isneginf(got_db)) or got_db.view(np.uint32) == want_db.view(np.uint32), (k, got_db, want_db)
        assert bool(lv["is_speech"][k]) == L.det.is_speaking()

    def close(self, k, vad_final=None, ended=False):
        """The life of stream k is over (an end, or a reset when ended=False): check it whole, start the next one."""
        L = self.life[k]
        pcm = np.concatenate(L.pcm) if L.pcm else np.zeros(0, np.float32)
        v = self.orc.VoiceActivityDetector()
        st, _ = v.stream(pcm, self.flen, self.hop)
        assert_bit_equal(np.concatenate(L.vad) if L.vad else np.zeros(0, np.uint8), st, f"stream {k} vad")
        if self.n_mels:
            got = np.concatenate(L.lm) if L.lm else np.zeros((0, self.n_mels), np.float32)
            assert_logmel_close(got, self.orc.logmel(pcm, self.orc.default_feat_config(self.n_mels)), f"stream {k} logmel")
        if vad_final is not None:
            assert (vad_final["state"], vad_final["speech_frames"]) == (v.state(), v.speech_frame_count()), k
            assert np.float32(vad_final["smoothed"]).view(np.uint32) == np.float32(v.smoothed_energy()).view(np.uint32), k
        if self.wire is not None and self.wire[0]:
            events, segs = _oracle_events(self.orc, st, L.frames, self.hop)
            if ended and len(st) and st[-1] == SPEECH:                # the end closes the open segment
                e = events[-1]
                events[-1] = (e[0], e[1], e[2] + 1, False, e[4], e[5])
            assert L.records == events, (k, L.records, events)
            want = self.orc.vad_gate(pcm, None, segs, self.hop)[0]
            got = np.concatenate(L.payload) if L.payload else np.zeros(0, np.int16)
            assert_bit_equal(got, self.orc.pcm16_encode(want), f"stream {k} gated payload")
            if ended:
                assert sum(r[1] for r in L.records) == sum(r[2] for r in L.records) == len(segs)
        self.closed += 1
        self.life[k] = _Life(self.orc, self.rate)

    def reset(self, ids):
        self.ses.reset_streams(ids)
        for k in set(ids) & self.check:
            self.close(k)

    def finish(self, last):
        for k in sorted(self.check):
            self.close(k, None if k in self.just_ended else last["vad_final"][k])


def _ragged_counts(rng, S, max_frames, ch, t):
    """Per stream: 0, one frame, the maximum, or anything between (seeded)."""
    pick = rng.integers(0, 6, S)
    n = rng.integers(0, max_frames + 1, S)
    n = np.where(pick == 0, 0, np.where(pick == 1, 1, np.where(pick == 2, max_frames, n)))
    return [int(v) * ch for v in n]


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rate,fmt,ch,max_frames", [(48000, "f32", 1, 960), (44100, "f32", 1, 882), (16000, "f32", 1, 320),
                                                     (32000, "f32", 1, 640), (48000, "i16", 2, 960)])
def test_ragged_ticks_match_reference_objects(af, orc, rate, fmt, ch, max_frames):
    rng = np.random.default_rng(rate + ch)
    S = 5
    h = Harness(af, orc, S, rate, ch, fmt, max_tick=max_frames * ch)
    for t in range(40):
        r = h.tick(_ragged_counts(rng, S, max_frames, ch, t))
    h.finish(r)


@pytest.mark.gpu
@pytest.mark.parametrize("rate", [48000, 44100, 16000])
@pytest.mark.parametrize("residual,before", [(0, "flush"), (127, "flush"), (127, "last_tick")])
def test_end_of_stream_equals_batch_path(af, orc, rate, residual, before):
    """Whole streams pushed raggedly with end on the last tick of max_tick_samples: process(all) + flush, and af_batch_run.
    `residual` is left over before the flush, or (the capacity case) before the full last tick: 127 + max_tick_samples
    frames then complete ceil(1087 / 128) = 9 chunks at once."""
    S, max_frames = 3, 960
    rng = np.random.default_rng(residual + rate + len(before))
    xs = [_source(orc, 40 + i, 0.7 + 0.13 * i, rate, 1, "f32") for i in range(S)]
    extra = max_frames if before == "last_tick" else 0
    xs = [x[: (len(x) // 128 - 8) * 128 + residual + extra] for x in xs]
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=80)), S, rate, 1, af.AF_FMT_F32, max_tick_samples=max_frames)
    got = [dict(pcm=[], lm=[], vad=[]) for _ in range(S)]
    pos = [0] * S
    finals = [None] * S
    while not all(finals):
        counts, end = [0] * S, [False] * S
        for k in range(S):
            if finals[k] is not None:
                continue
            left = len(xs[k]) - pos[k]
            if left == max_frames:
                n = max_frames
            elif left < 2 * max_frames:
                n = left - max_frames                                  # so that the last tick is a full one
            else:
                n = int(rng.integers(0, max_frames + 1))
            counts[k], end[k] = n, pos[k] + n == len(xs[k])
        r = ses.push_streams([xs[k][pos[k]:pos[k] + counts[k]] for k in range(S)], end)
        for k in range(S):
            pos[k] += counts[k]
            if finals[k] is None:
                got[k]["pcm"].append(r["pcm"][k]); got[k]["lm"].append(r["logmel"][k]); got[k]["vad"].append(r["vad"][k])
                if end[k]:
                    assert counts[k] == max_frames                            # the capacity case: a full tick, then the flush
                    finals[k] = r["vad_final"][k]
    batch = af.Pipeline(af.pipeline_config(n_mels=80)).run_host([(x, rate, 1) for x in xs])
    for k in range(S):
        ref = orc.pipeline_stream(xs[k], 1, rate, orc.default_feat_config(80), orc.default_vad_config())
        pcm = np.concatenate(got[k]["pcm"])
        assert_bit_equal(pcm, ref["pcm"], f"{k} pcm")
        assert_bit_equal(pcm, batch[k]["pcm"], f"{k} pcm vs batch")
        assert_bit_equal(np.concatenate(got[k]["vad"]), ref["vad"], f"{k} vad")
        assert_bit_equal(np.concatenate(got[k]["vad"]), batch[k]["vad"], f"{k} vad vs batch")
        assert_logmel_close(np.concatenate(got[k]["lm"]), ref["logmel"], f"{k} logmel")
        assert finals[k]["state"] == ref["vad_final"]["state"]
        assert finals[k]["speech_frames"] == ref["vad_final"]["speech_frames"]
        assert np.float32(finals[k]["smoothed"]).view(np.uint32) == np.float32(ref["vad_final"]["smoothed"]).view(np.uint32)


@pytest.mark.gpu
def test_slot_reuse_after_end_and_reset(af, orc):
    """An ended slot and reset slots serve new utterances from their first sample; the other streams go on bit-exact."""
    rng = np.random.default_rng(11)
    S = 6
    h = Harness(af, orc, S, 44100, max_tick=882, wire=(True, af.AF_MEM_HOST))
    for t in range(45):
        end = [False] * S
        if t in (10, 30):
            end[1] = True
        if t == 20:
            end[4] = True
        if t == 15:
            h.reset([2, 3, 2])                                         # several slots at once, one of them listed twice
        if t == 25:
            h.reset([3])
            h.reset([3])                                               # reset twice before its next push
        r = h.tick([int(n) for n in rng.integers(300, 1300, S) % 883], end)
    assert h.closed >= 6
    h.finish(r)


@pytest.mark.gpu
@pytest.mark.parametrize("wire_mem", ["host", "device"])
def test_lockstep_unchanged(af, orc, wire_mem):
    """push_streams with equal counts is the lockstep tick (same outputs, records and launches); push after divergence is
    push_streams with equal counts; reset restores lockstep."""
    from audioflow import synth
    S, tick, rate = 4, 960, 48000
    mem = af.AF_MEM_HOST if wire_mem == "host" else af.AF_MEM_DEVICE
    xs = [synth.stream(200 + i, 2.0, rate, 1)[: tick * 60] for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    plain = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    a.enable_wire(gate=True, mem=mem)
    b.enable_wire(gate=True, mem=mem)

    def launches(fn):
        l0 = af.kernel_launch_count()
        out = fn()
        return out, af.kernel_launch_count() - l0

    for t in range(12):
        x = np.stack([xx[t * tick:(t + 1) * tick] for xx in xs])
        ra, la = launches(lambda: a.push(x))
        rb, lb = launches(lambda: b.push_streams(list(x)))
        _, lp = launches(lambda: plain.push(x))
        assert la == lb == lp + 1                                      # the wire kernel on top of the plain tick
        if t > 0:
            assert lp == 4                                             # ingest+resample, fused (2), VAD scan
        for k in range(S):
            assert_bit_equal(ra["pcm"][k], rb["pcm"][k]); assert_bit_equal(ra["vad"][k], rb["vad"][k])
            assert_bit_equal(ra["logmel"][k], rb["logmel"][k])
        wa, wb = a.wire(), b.wire()
        assert wa["first_frame"] == wb["first_frame"] and list(wa["first_frames"]) == [wa["first_frame"]] * S
        for ga, gb in zip(wa["streams"], wb["streams"]):
            assert {k: v for k, v in ga.items() if k not in ("pcm16", "base64")} == \
                   {k: v for k, v in gb.items() if k not in ("pcm16", "base64")}
            if mem == af.AF_MEM_HOST:
                assert_bit_equal(ga["pcm16"], gb["pcm16"])
                assert ga["base64"] == gb["base64"]
    # divergence, then plain pushes on the diverged session, checked against the reference objects
    h = Harness(af, orc, S, rate, max_tick=tick)
    h.tick([960, 0, 500, 960])
    per_stream = 0
    for t in range(8):
        x = np.stack(h.samples([tick] * S))
        r = h.ses.push(x)                                              # Session.push on the diverged session
        per_stream += "n_pcm" in r                                     # the streams emitted different counts
        h.tick([tick] * S, xs=list(x), result=_as_streams(r, S))
    assert per_stream > 0
    # reset: lockstep again, same launches as a fresh session
    h.ses.reset()
    fresh = af.Session(h.pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    for t in range(3):
        x = np.stack([xx[t * tick:(t + 1) * tick] for xx in xs])
        r1, l1 = launches(lambda: h.ses.push_streams(list(x)))
        r2, l2 = launches(lambda: fresh.push(x))
        assert l1 == l2
        for k in range(S):
            assert_bit_equal(r1["pcm"][k], r2["pcm"][k]); assert_bit_equal(r1["vad"][k], r2["vad"][k])


def _as_streams(r, S):
    """Session.push's result in the per-stream form (it already has that form when the streams' counts differed)."""
    if "n_pcm" in r:
        return r
    return {"pcm": list(r["pcm"]), "logmel": list(r["logmel"]), "vad": list(r["vad"]),
            "n_pcm": np.full(S, r["pcm"].shape[1], np.uint32), "n_feat": np.full(S, r["logmel"].shape[1], np.uint32),
            "n_vad": np.full(S, r["vad"].shape[1], np.uint32), "vad_final": r["vad_final"]}


@pytest.mark.gpu
@pytest.mark.parametrize("gate", [False, True])
@pytest.mark.parametrize("wire_mem", ["host", "device"])
def test_wire_on_ragged_sessions(af, orc, gate, wire_mem):
    rng = np.random.default_rng(7 + gate)
    S = 5
    mem = af.AF_MEM_HOST if wire_mem == "host" else af.AF_MEM_DEVICE
    h = Harness(af, orc, S, 48000, max_tick=960, wire=(gate, mem))
    for t in range(50):
        end = [bool(rng.random() < 0.06) for _ in range(S)]
        r = h.tick(_ragged_counts(rng, S, 960, 1, t), end)
    assert h.closed >= 3
    h.finish(r)


@pytest.mark.gpu
def test_levels_on_ragged_ticks(af, orc):
    rng = np.random.default_rng(3)
    S = 4
    h = Harness(af, orc, S, 48000, max_tick=960, levels=True)
    for t in range(40):
        end = [bool(rng.random() < 0.05) for _ in range(S)]
        r = h.tick(_ragged_counts(rng, S, 960, 1, t), end)
    h.finish(r)


@pytest.mark.gpu
def test_rings_available_equals_push_streams(af, orc):
    """Uneven producers and empty rings: push_rings_available pushes what each ring holds (up to max, whole frames) and
    equals push_streams of the same samples; a partial frame stays in its ring."""
    S, ch, rate, mx = 4, 2, 48000, 1920
    xs = [_source(orc, 500 + i, 1.0, rate, ch, "f32") for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    ringed = af.Session(pipe, S, rate, ch, af.AF_FMT_F32, max_tick_samples=mx)
    direct = af.Session(pipe, S, rate, ch, af.AF_FMT_F32, max_tick_samples=mx)
    rings = [af.RingBuffer(8192) for _ in range(S)]
    fed, taken = [0] * S, [0] * S
    rng = np.random.default_rng(9)
    for t in range(30):
        for k in range(S):
            if k == 3 and t % 4:                                       # a stalled producer: its ring is often empty
                continue
            n = int(rng.integers(0, 1500))
            fed[k] += rings[k].write(xs[k][fed[k]:fed[k] + n])
        avail = [r.available() for r in rings]
        end = [t == 29] * S
        a = ringed.push_rings_available(rings, mx, end)
        want = [min(mx, v) // ch * ch for v in avail]
        assert [r.available() for r in rings] == [v - w for v, w in zip(avail, want)]   # odd leftovers stay
        b = direct.push_streams([xs[k][taken[k]:taken[k] + want[k]] for k in range(S)], end)
        for k in range(S):
            taken[k] += want[k]
            for key in ("pcm", "logmel", "vad"):
                assert_bit_equal(a[key][k], b[key][k], f"tick {t} {key} {k}")
        assert list(a["n_pcm"]) == list(b["n_pcm"])
    with pytest.raises(BufferError):                                   # max above max_tick_samples: nothing consumed
        before = [r.available() for r in rings]
        ringed.push_rings_available(rings, mx + ch)
    assert [r.available() for r in rings] == before


@pytest.mark.gpu
def test_errors_leave_the_session_untouched(af, orc):
    rng = np.random.default_rng(21)
    S, ch = 3, 2
    h = Harness(af, orc, S, 48000, ch, "f32", max_tick=960 * ch)
    L = af.load_library()
    u32p = C.POINTER(C.c_uint32)

    def short_rows(push):
        """Output rows too short for the largest stream's outputs: AF_ERR_CAPACITY, nothing changes."""
        pcm, lm, vad = np.zeros((S, 1024), np.float32), np.zeros((S, 16 * 80), np.float32), np.zeros((S, 16), np.uint8)
        for short in ("pcm", "logmel", "vad"):
            o = af.OutputsC(pcm.ctypes.data, 8 if short == "pcm" else 1024, lm.ctypes.data, 10 if short == "logmel" else 16 * 80,
                            vad.ctypes.data, 0 if short == "vad" else 16, None, 0, None)
            rc = push(C.byref(o))
            assert rc == af.AF_ERR_CAPACITY, (short, rc)

    for t in range(30):
        if t == 0:
            # the lockstep tick (every stream at the common position, equal counts): one tick so that the next completes
            # frames, then its own checks
            h.tick([960 * ch] * S)
            buf = np.zeros((S, 960 * ch), np.float32)
            short_rows(lambda o: L.af_session_push(h.ses._h, buf.ctypes.data, buf.shape[1], buf.shape[1], af.AF_MEM_HOST,
                                                   o, None, None, None))
        if t % 5 == 2:
            buf = np.zeros((S, 2000 * ch), np.float32)
            for counts, stride, status in (([961 * ch, 2, 2], buf.shape[1], af.AF_ERR_CAPACITY),   # above max_tick_samples
                                           ([3, 2, 2], buf.shape[1], af.AF_ERR_INVALID),           # a partial frame
                                           ([400, 600, 2], 500, af.AF_ERR_INVALID)):               # in_stride too small
                c = np.array(counts, np.uint32)
                rc = L.af_session_push_streams(h.ses._h, buf.ctypes.data, stride, c.ctypes.data_as(u32p), None,
                                               af.AF_MEM_HOST, None, None, None, None)
                assert rc == status, (counts, rc)
            assert L.af_session_push_streams(h.ses._h, buf.ctypes.data, buf.shape[1], None, None, af.AF_MEM_HOST,
                                             None, None, None, None) == af.AF_ERR_INVALID      # null counts
            with pytest.raises(ValueError):
                h.ses.reset_streams([1, S])                            # out of range: no stream is reset
            with pytest.raises(BufferError):
                h.ses.push_streams([np.zeros(962 * ch, np.float32)] * S)
            # the session has diverged: the per-stream plan checks
            c = np.full(S, 960 * ch, np.uint32)
            short_rows(lambda o: L.af_session_push_streams(h.ses._h, buf.ctypes.data, buf.shape[1], c.ctypes.data_as(u32p), None,
                                                           af.AF_MEM_HOST, o, None, None, None))
        end = [bool(rng.random() < 0.05) for _ in range(S)]
        r = h.tick(_ragged_counts(rng, S, 960, ch, t), end)
    h.finish(r)


@pytest.mark.gpu
def test_scale_1024_streams(af, orc):
    """1024 streams at 48 kHz, counts jittering around 960, about 1 % of the slots ending (and restarting) per tick; a
    seeded sample of 32 streams is checked against the oracle over 50 ticks."""
    S = 1024
    rng = np.random.default_rng(1024)
    check = sorted(int(k) for k in rng.choice(S, 32, replace=False))
    h = Harness(af, orc, S, 48000, max_tick=1440, check=check, seconds=4.0)
    for t in range(50):
        counts = [int(n) for n in rng.integers(480, 1441, S)]
        end = list(rng.random(S) < 0.01)
        r = h.tick(counts, end)
    h.finish(r)


def test_push_streams_arguments_are_checked_before_the_library():
    """No GPU: the rows of a ragged tick and the end flags are validated in Python before anything is pushed."""
    import audioflow as af
    buf, counts = af.stream_rows([np.ones(3, np.float32), np.zeros(0, np.float32), np.arange(6, dtype=np.float32)], 3, 1,
                                 np.float32)
    assert list(counts) == [3, 0, 6] and buf.shape == (3, 8)
    assert list(buf[2, :6]) == list(range(6)) and not buf[1].any()
    with pytest.raises(ValueError):
        af.stream_rows([np.ones(3)], 2, 1, np.float32)                 # one array per stream
    with pytest.raises(ValueError):
        af.stream_rows([np.ones(4), np.ones((2, 2))], 2, 1, np.float32)  # rows are 1-D interleaved samples
    with pytest.raises(ValueError):
        af.stream_rows([np.ones(4), np.ones(3)], 2, 2, np.float32)     # a partial stereo frame
    with pytest.raises(ValueError):
        af.end_flags([True], 2)
    assert af.end_flags(None, 2) is None and list(af.end_flags([True, 0], 2)) == [1, 0]
