"""Sessions of mixed capture formats (af_session_create_formats, af_session_restart_streams).  Stream k of such a session
must behave exactly like a one-stream af_session_create session of its current format pushed the same ticks, and like
the reference objects of that format: PCM, VAD states, detector states and wire payloads bit-exact against the oracle,
log-mel within assert_logmel_close, and everything (log-mel included) bitwise equal to the single-format session."""
import ctypes as C

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal
from test_session_streams_gpu import Harness, _Life, _as_streams, _source

# (sample_rate, channels, max_tick_samples): 20 ms of every capture device, plus 40 ms of 48 kHz stereo
FORMATS = [(48000, 1, 960), (48000, 2, 1920), (44100, 1, 882), (44100, 2, 1764), (32000, 1, 640), (22050, 1, 441),
           (16000, 1, 320)]


class Mixed(Harness):
    """Harness over a mixed session: every checked stream has reference objects of its own rate and channel count and,
    with twins=True, a one-stream af_session_create session of its format that is pushed the same ticks."""

    def __init__(self, af, orc, formats, stream_format, fmt="f32", n_mels=80, check=None, wire=None, levels=False,
                 twins=True, seconds=6.0):
        self.af, self.orc, self.S, self.fmt = af, orc, len(stream_format), fmt
        self.rate = 16000                  # (Harness.close starts a life at self.rate; close() below replaces it)
        self.n_mels, self.flen, self.hop = n_mels, 400, 160
        self._cache = {}
        self.sfmt = af.AF_FMT_I16 if fmt == "i16" else af.AF_FMT_F32
        self.formats, self.seconds = formats, seconds
        self.pipe = af.Pipeline(af.pipeline_config(n_mels=n_mels))
        self.ses = af.Session.formats(self.pipe, formats, stream_format, self.sfmt)
        self.check = set(range(self.S)) if check is None else set(check)
        self.sf = [int(f) for f in stream_format]
        self.src = [self._src(k) for k in range(self.S)]
        self.cur = [0] * self.S
        self.life = {k: _Life(orc, self.rate_of(k)) for k in self.check}
        self.wire, self.levels = wire, levels
        self.twins = {k: self._twin(k) for k in self.check} if twins else {}
        if wire is not None:
            self.ses.enable_wire(gate=wire[0], mem=wire[1])
        if levels:
            self.ses.enable_levels()
        self.closed, self.just_ended = 0, set()

    def rate_of(self, k):
        return self.formats[self.sf[k]][0]

    def ch_of(self, k):
        return self.formats[self.sf[k]][1]

    def _src(self, k):
        if k in self.check:
            return _source(self.orc, 300 + k, self.seconds, self.rate_of(k), self.ch_of(k), self.fmt)
        if self.sf[k] not in self._cache:                            # unchecked streams share one source per format
            self._cache[self.sf[k]] = _source(self.orc, 299, self.seconds, self.rate_of(k), self.ch_of(k), self.fmt)
        return self._cache[self.sf[k]]

    def _twin(self, k):
        r, ch, m = self.formats[self.sf[k]]
        t = self.af.Session(self.pipe, 1, r, ch, self.sfmt, max_tick_samples=m)
        if self.wire is not None:
            t.enable_wire(gate=self.wire[0], mem=self.af.AF_MEM_HOST)
        return t

    def _mono(self, x):
        # Harness.tick converts the checked streams in ascending order; tick() queued their channel counts
        return self.orc.to_mono(self.orc.i16_to_f32(x) if self.fmt == "i16" else np.asarray(x, np.float32), next(self._chs))

    def ragged(self, rng):
        """Per stream a count of its own format: 0, one frame, its bound, or anything between."""
        out = []
        for k in range(self.S):
            _, ch, m = self.formats[self.sf[k]]
            pick, n = int(rng.integers(0, 6)), int(rng.integers(0, m // ch + 1))
            out.append((0 if pick == 0 else 1 if pick == 1 else m // ch if pick == 2 else n) * ch)
        return out

    def tick(self, counts, end=None, xs=None, result=None):
        if xs is None:
            xs = self.samples(counts)
        r = result if result is not None else self.ses.push_streams(xs, end)
        w = self.ses.wire() if (self.wire is not None and self.twins) else None
        for k, t in self.twins.items():
            fin = end is not None and bool(end[k])
            rt = t.push_streams([xs[k]], [fin])
            for key in ("pcm", "logmel", "vad"):
                assert_bit_equal(r[key][k], rt[key][0], f"stream {k} {key} vs its one-format session")
            for key in ("n_pcm", "n_feat", "n_vad"):
                assert int(r[key][k]) == int(rt[key][0]), (k, key)
            assert r["vad_final"][k] == rt["vad_final"][0], k
            if w is not None:
                wt = t.wire()
                assert int(w["first_frames"][k]) == wt["first_frame"], k
                a, b = w["streams"][k], wt["streams"][0]
                assert {q: v for q, v in a.items() if q not in ("pcm16", "base64")} == \
                       {q: v for q, v in b.items() if q not in ("pcm16", "base64")}, k
                if a["pcm16"] is not None:
                    assert_bit_equal(a["pcm16"], b["pcm16"]); assert a["base64"] == b["base64"]
        self._chs = iter([self.ch_of(k) for k in sorted(self.check)])
        return super().tick(counts, end, xs, r)

    def close(self, k, vad_final=None, ended=False):
        super().close(k, vad_final, ended)
        self.life[k] = _Life(self.orc, self.rate_of(k))

    def restart(self, ids, fmts):
        """af_session_restart_streams: the listed streams start afresh in new formats (a stream that has pushed since
        its last start is checked whole first)."""
        self.ses.restart_streams(ids, fmts)
        for k, f in zip(ids, fmts):
            live = k in self.check and self.life[k].pcm
            self.sf[k] = int(f)
            if live:
                self.close(k)
            elif k in self.check:
                self.life[k] = _Life(self.orc, self.rate_of(k))
            self.src[k], self.cur[k] = self._src(k), 0
            if k in self.twins:
                self.twins[k] = self._twin(k)


def _launches(af, fn):
    l0 = af.kernel_launch_count()
    out = fn()
    return out, af.kernel_launch_count() - l0


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "i16"])
def test_ragged_mixed_ticks(af, orc, fmt):
    """Seven formats in one session (two streams of 44.1 kHz stereo), ragged counts, the odd end."""
    rng = np.random.default_rng(5 if fmt == "f32" else 6)
    h = Mixed(af, orc, FORMATS, [0, 1, 2, 3, 4, 5, 6, 3], fmt)
    for t in range(36):
        end = [bool(rng.random() < 0.04) for _ in range(h.S)]
        r = h.tick(h.ragged(rng), end)
    h.finish(r)


@pytest.mark.gpu
def test_ends_and_restarts_in_other_formats(af, orc):
    """Ends with residuals 0 and 127 followed by restarts in other formats, and restarts in the middle of a stream (no
    flush); every next life matches fresh reference objects and a fresh one-format session."""
    S = 6
    h = Mixed(af, orc, FORMATS, [0, 2, 3, 6, 1, 4], wire=(True, af.AF_MEM_HOST))
    rng = np.random.default_rng(17)
    plan = {6: (0, 0), 9: (1, 127), 13: (2, 0), 16: (4, 127)}        # tick: (stream, residual before the flush)
    frames = [0] * S                                                 # frames pushed in the stream's current life
    for t in range(30):
        counts, end = h.ragged(rng), [False] * S
        if t in plan:
            k, res = plan[t]
            ch = h.ch_of(k)
            counts[k] = ((res - frames[k]) % 128) * ch               # leaves `res` frames for the flush
            end[k] = True
        for k in range(S):
            frames[k] += counts[k] // h.ch_of(k)
        r = h.tick(counts, end)
        if t in plan:
            k = plan[t][0]
            h.restart([k], [(h.sf[k] + 3) % len(FORMATS)])          # the freed slot serves a caller with another device
            frames[k] = 0
        if t in (11, 20):
            ids = [5, 3] if t == 11 else [0]
            h.restart(ids, [(h.sf[k] + 1) % len(FORMATS) for k in ids])   # mid-stream: nothing is flushed
            for k in ids:
                frames[k] = 0
    assert h.closed >= 7
    h.finish(r)


@pytest.mark.gpu
def test_plan_sharing(af, orc):
    """Groups of streams in one format at one position (their 44.1 kHz fraction slice shared) next to streams of the
    same format at other positions, and groups whose members split apart and meet again after a restart."""
    S = 12
    sf = [2] * 8 + [1, 1, 3, 3]
    h = Mixed(af, orc, FORMATS, sf)
    rng = np.random.default_rng(29)
    for t in range(30):
        n_a, n_b, n_c = int(rng.integers(0, 883)), int(rng.integers(0, 961)) * 2, int(rng.integers(0, 883)) * 2
        counts = [n_a] * 6 + [882, 441 if t % 3 else 0] + [n_b, n_b, n_c, n_c]
        if t == 0:
            counts[6] = 100                                          # 6 and 7 at other positions than 0-5
        if t == 10:
            counts[5] = 0                                            # 5 leaves the group ...
        if t == 20:
            h.restart([0, 1, 2], [2, 2, 2])                          # ... 0-2 restart together, one group again
        r = h.tick(counts)
    h.finish(r)


@pytest.mark.gpu
@pytest.mark.parametrize("gate", [False, True])
@pytest.mark.parametrize("wire_mem", ["host", "device"])
def test_wire_and_levels_on_mixed_sessions(af, orc, gate, wire_mem):
    rng = np.random.default_rng(40 + 2 * gate + (wire_mem == "host"))
    mem = af.AF_MEM_HOST if wire_mem == "host" else af.AF_MEM_DEVICE
    h = Mixed(af, orc, FORMATS, [0, 1, 2, 3, 6, 5], wire=(gate, mem), levels=True)
    for t in range(36):
        end = [bool(rng.random() < 0.05) for _ in range(h.S)]
        r = h.tick(h.ragged(rng), end)
    h.finish(r)


@pytest.mark.gpu
def test_push_on_a_mixed_session(af, orc):
    """Session.push (af_session_push) with one count every stream's channels divide: the per-stream form of the result."""
    h = Mixed(af, orc, FORMATS, [0, 1, 2, 3, 4, 5, 6])
    for t in range(12):
        n = (320, 160, 0)[t % 3]                                     # whole stereo frames, within every bound
        x = np.stack(h.samples([n] * h.S))
        r = h.ses.push(x)
        if n:
            assert "n_pcm" in r                                      # the rates differ: per-stream outputs
        else:                                                        # nothing emitted: equal counts, the [S, 0] form
            assert "n_pcm" not in r and r["pcm"].shape == (h.S, 0)
        h.tick([n] * h.S, xs=list(x), result=_as_streams(r, h.S))
    h.finish(r)


@pytest.mark.gpu
def test_rings_on_a_mixed_session(af, orc):
    """push_rings takes exactly n from every ring; push_rings_available clamps every stream to its own format's bound and
    rounds to whole frames of its own channels.  Both equal push_streams of the same samples on a twin session."""
    fmts = [(48000, 2, 1920), (16000, 1, 320), (44100, 1, 882), (48000, 1, 960)]
    sf = [0, 1, 2, 3, 0]
    S = len(sf)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    ringed = af.Session.formats(pipe, fmts, sf)
    direct = af.Session.formats(pipe, fmts, sf)
    xs = [_source(orc, 700 + k, 1.5, fmts[f][0], fmts[f][1], "f32") for k, f in enumerate(sf)]
    rings = [af.RingBuffer(16384) for _ in range(S)]
    fed, taken = [0] * S, [0] * S
    rng = np.random.default_rng(13)

    def compare(a, b, t):
        for k in range(S):
            for key in ("pcm", "logmel", "vad"):
                assert_bit_equal(a[key][k], b[key][k], f"tick {t} {key} {k}")
        assert list(a["n_pcm"]) == list(b["n_pcm"])

    for t in range(24):
        for k in range(S):
            n = int(rng.integers(0, 2500)) if k != 4 or t % 3 == 0 else 0
            fed[k] += rings[k].write(xs[k][fed[k]:fed[k] + n])
        if t % 4 == 0 and min(r.available() for r in rings) >= 320:
            a = _as_streams(ringed.push_rings(rings, 320), S)
            b = direct.push_streams([xs[k][taken[k]:taken[k] + 320] for k in range(S)])
            taken = [v + 320 for v in taken]
            compare(a, b, t)
            continue
        avail = [r.available() for r in rings]
        a = ringed.push_rings_available(rings, 1920)
        want = [min(1920, fmts[f][2], v) // fmts[f][1] * fmts[f][1] for f, v in zip(sf, avail)]
        assert [r.available() for r in rings] == [v - w for v, w in zip(avail, want)]
        b = direct.push_streams([xs[k][taken[k]:taken[k] + want[k]] for k in range(S)])
        taken = [v + w for v, w in zip(taken, want)]
        compare(a, b, t)
    before = [r.available() for r in rings]
    with pytest.raises(BufferError):                                 # above the largest bound (1920 + one stereo frame)
        ringed.push_rings_available(rings, 1922)
    with pytest.raises(ValueError):                                  # not whole frames of the stereo streams
        ringed.push_rings(rings, 3)
    assert [r.available() for r in rings] == before


@pytest.mark.gpu
def test_single_format_equivalence(af, orc):
    """af_session_create_formats with one format is af_session_create: the lockstep tick, the same launches, bitwise
    outputs, on equal and on ragged ticks."""
    from audioflow import synth
    S, tick, rate = 4, 960, 48000
    xs = [synth.stream(200 + i, 2.0, rate, 1)[: tick * 40] for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session.formats(pipe, [(rate, 1, tick)], [0] * S)
    a.enable_wire(gate=True); b.enable_wire(gate=True)
    rng = np.random.default_rng(3)
    pos = [0] * S
    for t in range(24):
        if t < 8 or t >= 20:
            x = np.stack([xx[pos[k]:pos[k] + tick] for k, xx in enumerate(xs)])
            pos = [p + tick for p in pos]
            ra, la = _launches(af, lambda: a.push(x))
            rb, lb = _launches(af, lambda: b.push(x))
            assert la == lb and "n_pcm" not in ra and "n_pcm" not in rb   # the lockstep tick
            ra, rb = _as_streams(ra, S), _as_streams(rb, S)
        else:
            counts = [int(n) for n in rng.integers(0, tick + 1, S)]
            chunk = [xx[pos[k]:pos[k] + counts[k]] for k, xx in enumerate(xs)]
            pos = [p + n for p, n in zip(pos, counts)]
            ra, la = _launches(af, lambda: a.push_streams(chunk))
            rb, lb = _launches(af, lambda: b.push_streams(chunk))
            assert la == lb
        for k in range(S):
            for key in ("pcm", "logmel", "vad"):
                assert_bit_equal(ra[key][k], rb[key][k], f"tick {t} {key} {k}")
        assert ra["vad_final"] == rb["vad_final"]
        wa, wb = a.wire(), b.wire()
        assert list(wa["first_frames"]) == list(wb["first_frames"])
        for ga, gb in zip(wa["streams"], wb["streams"]):
            assert ga["base64"] == gb["base64"] and ga["n_samples"] == gb["n_samples"] and ga["ended"] == gb["ended"]
            assert_bit_equal(ga["pcm16"], gb["pcm16"])
        if t == 19:
            a.reset(); b.reset()                                     # lockstep again
            pos = [0] * S


@pytest.mark.gpu
def test_errors_leave_the_session_untouched(af, orc):
    L = af.load_library()
    u32p = C.POINTER(C.c_uint32)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))

    def create(formats, sf, n=2, sample_format=af.AF_FMT_F32):
        arr = (af.StreamFormatC * max(len(formats), 1))(*[af.StreamFormatC(*f) for f in formats])
        s = None if sf is None else (C.c_uint32 * n)(*sf)
        h = C.c_void_p()
        rc = L.af_session_create_formats(pipe._h, n, arr, len(formats), s, sample_format, C.byref(h))
        if rc == af.AF_OK:
            L.af_session_destroy(h)
        return rc

    good = (48000, 1, 0, 960)
    assert create([good], None) == af.AF_OK
    assert create([good, (16000, 2, 0, 640)], [1, 0]) == af.AF_OK
    assert create([], None) == af.AF_ERR_INVALID                                 # no format
    for bad in ((0, 1, 0, 960), (48000, 0, 0, 960), (48000, 1, 0, 0), (48000, 1, 1, 960)):
        assert create([good, bad], [0, 0]) == af.AF_ERR_INVALID, bad            # zero rate / channels / bound, pad
    assert create([good], [0, 1]) == af.AF_ERR_INVALID                          # stream_format out of range
    assert create([good], [0, 0], sample_format=7) == af.AF_ERR_INVALID
    assert create([good, (4000000, 1, 0, 960)], [0, 0]) == af.AF_ERR_RESAMPLING_FAILED   # a step past the chunk
    assert create([good, (48000, 1, 0, 1 << 20)], [0, 0]) == af.AF_ERR_INVALID  # does not fit a session tile

    rng = np.random.default_rng(21)
    h = Mixed(af, orc, FORMATS, [1, 6, 2, 0])
    for t in range(24):
        if t % 6 == 3:
            buf = np.zeros((h.S, 4000), np.float32)
            for counts, status in (([1920, 322, 0, 0], af.AF_ERR_CAPACITY),     # above stream 1's own bound (16 kHz, 320)
                                   ([1922, 0, 0, 0], af.AF_ERR_CAPACITY),       # above the stereo bound
                                   ([3, 0, 0, 0], af.AF_ERR_INVALID)):          # a partial stereo frame
                c = np.array(counts, np.uint32)
                rc = L.af_session_push_streams(h.ses._h, buf.ctypes.data, buf.shape[1], c.ctypes.data_as(u32p), None,
                                               af.AF_MEM_HOST, None, None, None, None)
                assert rc == status, (counts, rc)
            assert L.af_session_push(h.ses._h, buf.ctypes.data, buf.shape[1], 3, af.AF_MEM_HOST, None, None, None,
                                     None) == af.AF_ERR_INVALID                 # af_session_push: partial stereo frame
            ids, fm = np.array([0, 4], np.uint32), np.array([1, 1], np.uint32)
            assert L.af_session_restart_streams(h.ses._h, ids.ctypes.data_as(u32p), fm.ctypes.data_as(u32p), 2) == af.AF_ERR_INVALID
            ids, fm = np.array([0, 1], np.uint32), np.array([1, len(FORMATS)], np.uint32)
            assert L.af_session_restart_streams(h.ses._h, ids.ctypes.data_as(u32p), fm.ctypes.data_as(u32p), 2) == af.AF_ERR_INVALID
            rings = [af.RingBuffer(8192) for _ in range(h.S)]
            for rg in rings:
                rg.write(np.zeros(4000, np.float32))
            with pytest.raises(BufferError):
                h.ses.push_rings_available(rings, 1922)
            assert [rg.available() for rg in rings] == [4000] * h.S
        end = [bool(rng.random() < 0.05) for _ in range(h.S)]
        r = h.tick(h.ragged(rng), end)                              # bit-exact on: nothing changed
    h.finish(r)


@pytest.mark.gpu
def test_scale_1024_mixed_streams(af, orc):
    """1024 streams in the benchmark's mix (512 x 48 kHz, 256 x 44.1 kHz, 128 x 48 kHz stereo, 128 x 16 kHz), counts
    jittering around 20 ms, about 1 % of the slots ending and restarting in another format per tick; 32 streams checked."""
    fmts = [(48000, 1, 1440), (44100, 1, 1323), (48000, 2, 2880), (16000, 1, 480)]
    sf = [0] * 512 + [1] * 256 + [2] * 128 + [3] * 128
    rng = np.random.default_rng(1024)
    check = sorted(int(k) for k in rng.choice(1024, 32, replace=False))
    h = Mixed(af, orc, fmts, sf, check=check, twins=False, seconds=3.0)
    for t in range(40):
        counts = []
        for k in range(1024):
            _, ch, m = fmts[h.sf[k]]
            counts.append(int(rng.integers(m // ch // 3, m // ch + 1)) * ch)
        end = list(rng.random(1024) < 0.01)
        r = h.tick(counts, end)
        ended = [k for k in range(1024) if end[k]]
        h.restart(ended, [(h.sf[k] + 1 + int(rng.integers(0, 3))) % 4 for k in ended])
    h.finish(r)


# ---- no GPU -----------------------------------------------------------------------------------------------------------
def test_stream_format_layout():
    """af_stream_format is 12 bytes: rate at 0, channels at 4, pad at 6, bound at 8."""
    import audioflow as af
    F = af.StreamFormatC
    assert C.sizeof(F) == 12
    assert (F.sample_rate.offset, F.channels.offset, F.pad.offset, F.max_tick_samples.offset) == (0, 4, 6, 8)


def test_mixed_session_arguments_are_checked_before_the_library():
    """No GPU: a mixed session checks counts against each stream's own channels, and restart_streams its indices, in
    Python before the library is called (a session object with no library handle stands in)."""
    import audioflow as af
    s = af.Session.__new__(af.Session)
    s._setup(None, None, [(48000, 1, 960), (44100, 2, 1764)], np.array([0, 1, 1], np.uint32), af.AF_FMT_F32)
    assert list(s.stream_channels()) == [1, 2, 2] and s.rate is None and s.channels is None
    with pytest.raises(ValueError):                                  # 3 samples: a partial frame of streams 1 and 2
        s.push_streams([np.ones(4, np.float32), np.ones(4, np.float32), np.ones(3, np.float32)])
    with pytest.raises(ValueError):
        s.push(np.ones((3, 5), np.float32))
    with pytest.raises(ValueError):
        s.restart_streams([0, 3], [0, 0])                            # stream out of range
    with pytest.raises(ValueError):
        s.restart_streams([0], [2])                                  # format out of range
    with pytest.raises(ValueError):
        s.restart_streams([0, 1], [1])                               # one format per stream
    assert list(s.stream_format) == [0, 1, 1]                        # nothing changed
    one = af.Session.__new__(af.Session)
    one._setup(None, None, [(16000, 1, 320)], np.zeros(2, np.uint32), af.AF_FMT_F32)
    assert (one.rate, one.channels) == (16000, 1)
    s._h = None                                                      # (nothing to destroy)
    one._h = None
