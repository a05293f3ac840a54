"""Per-stream VAD configurations (af_batch_set_vad_configs, af_session_set_vad_configs): every caller's
VoiceActivityDetector::new(config) (vad.rs:21-43, 80-88) inside one batch or session.  Stream k must behave exactly like
a one-stream batch or session whose pipeline has its configuration, and like the oracle detector with that configuration:
states, energies, vad_final, levels and wire payloads bit-exact; PCM and log-mel unchanged by any configuration.  A change
between ticks is the oracle detector with its config replaced (_set_config) before the push's first frame."""
import ctypes as C
import math

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal
from test_session_formats_gpu import FORMATS, Mixed
from test_session_streams_gpu import _Life, _source
from test_session_wire_gpu import _oracle_events

SPEECH = 1


def _configs(af):
    """The range a server meets: the default, thresholds -35 / -60 / NaN (never speech), smoothing 0 (raw energy), 0.1,
    0.5, 1 (no memory) and 0.05 (too slow for the parallel scan: the sequential kernel), silence timeouts 0 / 1 / 5 / 40,
    minimum speech 0 / 1 / 10, and two mixtures."""
    V = af.VadConfig
    return [V(), V(threshold_db=-35.0), V(threshold_db=-60.0), V(threshold_db=math.nan), V(smoothing_factor=0.0),
            V(smoothing_factor=0.1), V(smoothing_factor=0.5), V(smoothing_factor=1.0), V(smoothing_factor=0.05),
            V(silence_timeout_frames=0), V(silence_timeout_frames=1), V(silence_timeout_frames=5),
            V(silence_timeout_frames=40), V(min_speech_frames=0), V(min_speech_frames=1), V(min_speech_frames=10),
            V(-60.0, 0.1, 5, 1), V(-35.0, 0.5, 40, 10)]


def _oc(orc, c):
    o = orc.default_vad_config()
    o.threshold_db, o.smoothing_factor = c.threshold_db, c.smoothing_factor
    o.silence_timeout_frames, o.min_speech_frames = c.silence_timeout_frames, c.min_speech_frames
    return o


def _set_config(det, oc):
    """The reference detector with its `config` field replaced between two detect calls, which is how the library
    defines a mid-stream change (DESIGN.md section 10).  The oracle's detector (orc_vad, oracle/oracle.c) starts with its
    orc_vad_config, so the configuration is overwritten in place and the state fields after it are kept;
    test_config_replacement_keeps_the_state pins that on a hand-worked sequence."""
    C.memmove(det._h, C.byref(oc), C.sizeof(oc))


def _levels_signal(seed, seconds, rate, ch=1):
    """Noise in stretches of four loudness classes (about -80, -58, -49 and -28 dB mean square): each threshold of
    _configs (-35, -50, -60) sees speech start and stop, and the EMA regimes differ."""
    rng = np.random.default_rng(seed)
    n = int(seconds * rate)
    seg = rng.integers(0, 4, n // 3000 + 1).repeat(3000)[:n]
    x = (np.choose(seg, [0.01, 0.035, 0.06, 0.2]).astype(np.float32) * rng.standard_normal(n).astype(np.float32))
    x = x.clip(-1, 1)
    return np.repeat(x, ch) if ch > 1 else x


def _launches(af, fn):
    l0 = af.kernel_launch_count()
    out = fn()
    return out, af.kernel_launch_count() - l0


def _run_batch(af, pipe, streams, cfgs="unset"):
    """A host batch over `streams` ((x, rate, ch) each): (per-stream results, kernel launches of the run)."""
    descs = [(x.ctypes.data, x.size, rate, ch, af.AF_FMT_F32) for x, rate, ch in streams]
    b = af.Batch(pipe, descs, af.AF_MEM_HOST)
    if cfgs != "unset":
        b.set_vad_configs(cfgs)
    out = b.alloc_host_outputs()
    _, n = _launches(af, lambda: b.run_host(out))
    return b.split(out), n


def _same_vad(g, r, what):
    assert_bit_equal(g["vad"], r["vad"], what + " vad")
    assert_bit_equal(g["energy"], r["energy"], what + " energy")
    assert g["vad_final"] == r["vad_final"], (what, g["vad_final"], r["vad_final"])


def _against_oracle(orc, g, x, ch, rate, oc, flen, hop, what):
    ref = orc.pipeline_stream(x, ch, rate, None, oc, flen, hop, "f32")
    assert_bit_equal(g["vad"], ref["vad"], what + " vad vs oracle")
    assert_bit_equal(g["energy"], ref["energy"], what + " energy vs oracle")
    f = g["vad_final"]
    assert (f["state"], f["speech_frames"]) == (ref["vad_final"]["state"], ref["vad_final"]["speech_frames"]), what
    assert np.float32(f["smoothed"]).view(np.uint32) == np.float32(ref["vad_final"]["smoothed"]).view(np.uint32), what


# ---- batches ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("framing", ["stft", "20ms"])
def test_batch_mixed_configs(af, orc, framing):
    """48 streams of 30 s at 44.1 and 48 kHz, one configuration each (alpha = 0.05 next to parallel-scan streams)."""
    cfgs = _configs(af)
    S = 48
    streams = [(_levels_signal(10 + k, 30.0, 44100 if k % 3 == 1 else 48000), 44100 if k % 3 == 1 else 48000, 1)
               for k in range(S)]
    per = [cfgs[k % len(cfgs)] for k in range(S)]
    kw = dict(n_mels=80) if framing == "stft" else dict(n_mels=0, vad_frame_len=320, vad_hop=320)
    flen, hop = (400, 160) if framing == "stft" else (320, 320)
    pipe = af.Pipeline(af.pipeline_config(**kw))
    plain, n_plain = _run_batch(af, pipe, streams)
    got, n_got = _run_batch(af, pipe, streams, per)
    # the sequential kernel after the parallel one in each stream group (about 32 MB: 6 streams) that holds one of the
    # three alpha = 0.05 streams (8, 26, 44)
    assert n_got == n_plain + 3
    for k, (x, rate, ch) in enumerate(streams):
        what = f"{framing} stream {k} ({per[k]})"
        assert_bit_equal(got[k]["pcm"], plain[k]["pcm"], what + " pcm")
        if framing == "stft":
            assert_bit_equal(got[k]["logmel"], plain[k]["logmel"], what + " logmel")
        _against_oracle(orc, got[k], x, ch, rate, _oc(orc, per[k]), flen, hop, what)
        one, _ = _run_batch(af, af.Pipeline(af.pipeline_config(vad=per[k], **kw)), [streams[k]])
        _same_vad(got[k], one[0], what + " vs one-stream batch")


@pytest.mark.gpu
def test_batch_long_streams_mixed_configs(af, orc):
    """Streams of more than 16384 frames take the many-CTA scan; each CTA reads its own stream's record (timeout, sync-point
    rule, warm-up).  Continuous speech across whole blocks (no sync point), flicker at block boundaries, and an alpha = 0.05
    stream that the sequential kernel takes next to them."""
    rng = np.random.default_rng(23)
    fs = 16000
    def noise(sec, a): return (a * rng.standard_normal(int(sec * fs))).astype(np.float32).clip(-1, 1)
    x1 = np.concatenate([noise(5, 1e-3), noise(200, 0.3), noise(40, 1e-3), noise(60, 0.056)])     # no sync point, flicker
    x2 = np.concatenate([noise(78, 1e-3), noise(10, 0.056), noise(150, 0.02), noise(30, 1e-3)])   # flicker at 81.92 s
    x3 = _levels_signal(3, 330.0, fs)
    x4 = _levels_signal(4, 280.0, fs)
    V = af.VadConfig
    per = [V(silence_timeout_frames=40), V(-35.0, 0.3, 1, 3), V(silence_timeout_frames=0, min_speech_frames=10),
           V(smoothing_factor=0.05), V(-60.0, 0.5, 5, 1)]
    streams = [(x, fs, 1) for x in (x1, x2, x3, x4)] + [(x3[:fs * 20], fs, 1)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=0))
    got, _ = _run_batch(af, pipe, streams, per)
    for k, (x, rate, ch) in enumerate(streams):
        assert len(got[k]["vad"]) > 16384 or k == 4
        _against_oracle(orc, got[k], x, ch, rate, _oc(orc, per[k]), 400, 160, f"long stream {k}")


@pytest.mark.gpu
def test_batch_identity(af, orc):
    """Every stream set to the pipeline's configuration, and None after a mixed set, give the unconfigured output bitwise
    with the same launches, on a host batch of several stream groups (each group's slice of the records must be its own)."""
    cfgs = _configs(af)
    S = 14
    streams = [(_levels_signal(60 + k, 60.0, 48000 if k % 2 else 44100), 48000 if k % 2 else 44100, 1) for k in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    descs = [(x.ctypes.data, x.size, rate, ch, af.AF_FMT_F32) for x, rate, ch in streams]
    b = af.Batch(pipe, descs, af.AF_MEM_HOST)
    assert sum(x.nbytes for x, _, _ in streams) > 4 * (32 << 20)        # several 32 MB stream groups

    def run():
        out = b.alloc_host_outputs()
        _, n = _launches(af, lambda: b.run_host(out))
        return b.split(out), n

    base, n0 = run()
    b.set_vad_configs([af.VadConfig()] * S)
    same, n1 = run()
    per = [cfgs[(3 * k + 1) % len(cfgs)] for k in range(S)]
    b.set_vad_configs(per)
    mixed, _ = run()
    b.set_vad_configs(None)
    back, n2 = run()
    assert n0 == n1 == n2
    for k, (x, rate, ch) in enumerate(streams):
        for r, what in ((same, "pipeline's config"), (back, "None after a mixed set")):
            for key in ("pcm", "logmel", "vad", "energy"):
                assert_bit_equal(r[k][key], base[k][key], f"{what} stream {k} {key}")
            assert r[k]["vad_final"] == base[k]["vad_final"]
        assert_bit_equal(mixed[k]["pcm"], base[k]["pcm"], f"mixed stream {k} pcm")
        assert_bit_equal(mixed[k]["logmel"], base[k]["logmel"], f"mixed stream {k} logmel")
        _against_oracle(orc, mixed[k], x, ch, rate, _oc(orc, per[k]), 400, 160, f"mixed stream {k}")


# ---- sessions ----------------------------------------------------------------------------------------------------------
class _ConfiguredOrc:
    """The oracle module with VoiceActivityDetector() built for one configuration (the harness builds default ones)."""

    def __init__(self, orc, oc):
        self._orc, self._oc = orc, oc

    def __getattr__(self, name):
        return getattr(self._orc, name)

    def VoiceActivityDetector(self, config=None):
        return self._orc.VoiceActivityDetector(self._oc)


class Configured(Mixed):
    """Mixed harness whose streams each have a VAD configuration: the reference objects use it, and every checked stream's
    twin is a one-stream session whose pipeline has it."""

    def __init__(self, af, orc, formats, stream_format, cfgs, **kw):
        self.cfgs = list(cfgs)
        super().__init__(af, orc, formats, stream_format, **kw)
        self.ses.set_vad_configs(range(self.S), self.cfgs)
        self.life = {k: _Life(self._orc_of(k), self.rate_of(k)) for k in self.check}

    def _orc_of(self, k):
        return _ConfiguredOrc(self.orc, _oc(self.orc, self.cfgs[k]))

    def _twin(self, k):
        r, ch, m = self.formats[self.sf[k]]
        pipe = self.af.Pipeline(self.af.pipeline_config(n_mels=self.n_mels, vad=self.cfgs[k]))
        t = self.af.Session(pipe, 1, r, ch, self.sfmt, max_tick_samples=m)
        t._pipe_ref = pipe
        if self.wire is not None:
            t.enable_wire(gate=self.wire[0], mem=self.af.AF_MEM_HOST)
        if self.levels:
            t.enable_levels()
        return t

    def tick(self, counts, end=None, xs=None, result=None):
        if xs is None:
            xs = self.samples(counts)
        r = self.ses.push_streams(xs, end)
        lv = self.ses.levels() if self.levels else None
        for k, t in self.twins.items():
            if lv is not None:                       # (Mixed.tick pushes the twins; their levels are read afterwards)
                t._lv_main = (lv["level_db"][k], lv["is_speech"][k])
        out = super().tick(counts, end, xs, r)
        if lv is not None:
            for k, t in self.twins.items():
                tl = t.levels()
                assert tl["level_db"][0].view(np.uint32) == t._lv_main[0].view(np.uint32), k
                assert bool(tl["is_speech"][0]) == bool(t._lv_main[1]), k
        return out

    def close(self, k, vad_final=None, ended=False):
        orc = self.orc
        self.orc = self._orc_of(k)                   # the life ends under the configuration it ran with
        try:
            super().close(k, vad_final, ended)
        finally:
            self.orc = orc

    def take_over(self, ids, fmts, cfgs):
        """A new caller takes each slot: restart in its format, then its configuration, before its first push."""
        self.restart(ids, fmts)
        self.ses.set_vad_configs(ids, cfgs)
        for k, c in zip(ids, cfgs):
            self.cfgs[k] = c
            if k in self.check:
                self.life[k] = _Life(self._orc_of(k), self.rate_of(k))
            if k in self.twins:
                self.twins[k] = self._twin(k)


@pytest.mark.gpu
@pytest.mark.parametrize("wire_mem", ["host", "device"])
def test_session_configs_per_slot(af, orc, wire_mem):
    """Ragged ticks of four formats, 1 % of the streams ending per tick and their slots taken over by callers with
    another format and configuration; gated wire output and levels on."""
    mem = af.AF_MEM_HOST if wire_mem == "host" else af.AF_MEM_DEVICE
    cfgs = _configs(af)
    S = 100
    rng = np.random.default_rng(70 + (wire_mem == "host"))
    sf = [k % 4 for k in range(S)]
    check = list(range(0, S, 7))
    h = Configured(af, orc, FORMATS[:4], sf, [cfgs[k % len(cfgs)] for k in range(S)], check=check,
                   wire=(True, mem), levels=True, seconds=8.0)
    n_taken = 0
    for t in range(40):
        end = [False] * S
        for k in rng.choice(S, 1, replace=False):
            end[int(k)] = True
        if t % 10 == 3:
            end[check[(t // 10) % len(check)]] = True                # a checked stream among them
        r = h.tick(h.ragged(rng), end)
        if t == 39:
            break
        ended = [k for k in range(S) if end[k]]
        new_cfg = [cfgs[int(rng.integers(0, len(cfgs)))] for _ in ended]
        h.take_over(ended, [(h.sf[k] + 1) % 4 for k in ended], new_cfg)
        n_taken += len(ended)
    assert n_taken >= 40 and h.closed >= 4
    h.finish(r)


@pytest.mark.gpu
def test_session_mid_stream_change(af, orc):
    """Configurations changed between ticks, in Speech and to a timeout below the stream's current silence count: the
    states, vad_final, wire records and the concatenated gated payload equal the oracle detector with _set_config
    applied before the push's first completed frame."""
    cfgs = _configs(af)
    S, rate, max_tick, flen, hop = 8, 48000, 960, 400, 160
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    ses = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=max_tick)
    ses.enable_wire(gate=True, mem=af.AF_MEM_HOST)
    src = [_source(orc, 500 + k, 5.0, rate, 1, "f32") for k in range(S)]
    rng = np.random.default_rng(91)
    det = [orc.VoiceActivityDetector() for _ in range(S)]
    pcm = [np.zeros(0, np.float32) for _ in range(S)]
    states = [[] for _ in range(S)]
    frames = [[] for _ in range(S)]
    payload = [[] for _ in range(S)]
    records = [[] for _ in range(S)]
    pos = [0] * S
    hard = 0                                                           # changes in Speech to a timeout below the count
    for t in range(150):
        if t >= 5 and t % 3 == 0:
            ids, new = [], []
            for k in range(S):
                d = det[k]
                if d.state() == SPEECH and d.silence_frames() >= 2:
                    ids.append(k); new.append(af.VadConfig(silence_timeout_frames=int(d.silence_frames()) - 1))
                    hard += 1
                elif rng.random() < 0.3:
                    ids.append(k); new.append(cfgs[int(rng.integers(0, len(cfgs)))])
            if ids:
                if len(ids) > 1:                                        # a stream listed twice: the last entry wins
                    ids, new = ids + [ids[0]], [cfgs[0]] + new[1:] + [new[0]]
                ses.set_vad_configs(ids, new)
                for k, c in zip(ids, new):
                    _set_config(det[k], _oc(orc, c))
        counts = [int(v) for v in rng.integers(0, max_tick + 1, S)]
        xs = [src[k][pos[k]:pos[k] + counts[k]] for k in range(S)]
        for k in range(S):
            pos[k] += counts[k]
        r = ses.push_streams(xs)
        w = ses.wire()
        for k in range(S):
            before = orc.num_frames(len(pcm[k]), flen, hop)
            pcm[k] = np.concatenate([pcm[k], r["pcm"][k]])
            T = orc.num_frames(len(pcm[k]), flen, hop) - before
            assert int(r["n_vad"][k]) == T
            want = np.array([det[k].detect(pcm[k][f * hop:f * hop + flen]) for f in range(before, before + T)], np.uint8)
            assert_bit_equal(r["vad"][k], want, f"tick {t} stream {k} states")
            states[k].append(want)
            frames[k].append(T)
            fin = r["vad_final"][k]
            assert (fin["state"], fin["speech_frames"]) == (det[k].state(), det[k].speech_frame_count()), (t, k)
            assert np.float32(fin["smoothed"]).view(np.uint32) == np.float32(det[k].smoothed_energy()).view(np.uint32)
            g = w["streams"][k]
            payload[k].append(g["pcm16"])
            records[k].append((before, g["started"], g["ended"], g["in_speech"], g["continued"], g["n_samples"]))
    assert hard >= 3
    for k in range(S):
        st = np.concatenate(states[k])
        events, segs = _oracle_events(orc, st, frames[k], hop)
        assert records[k] == events, k
        want = orc.vad_gate(pcm[k], None, segs, hop)[0]
        assert_bit_equal(np.concatenate(payload[k]), orc.pcm16_encode(want), f"stream {k} gated payload")


@pytest.mark.gpu
def test_session_pipeline_config_everywhere_changes_nothing(af):
    """cfg5 shape (1024 x 20 ms at 48 kHz): every stream set to the pipeline's configuration keeps the lockstep tick with
    its 4 launches and stays bitwise equal to an untouched session."""
    from audioflow import synth
    S, tick = 1024, 960
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    a.set_vad_configs(range(S), [af.VadConfig()] * S)
    base = [synth.stream(700 + i, 1.0, 48000, 1) for i in range(8)]
    for t in range(12):
        x = np.stack([base[k % 8][t * tick:(t + 1) * tick] for k in range(S)])
        ra, la = _launches(af, lambda: a.push(x))
        rb, lb = _launches(af, lambda: b.push(x))
        assert la == lb
        if t > 0:
            assert la == 4
        assert "n_pcm" not in ra                                      # the lockstep form
        for key in ("pcm", "logmel", "vad"):
            assert_bit_equal(ra[key], rb[key], f"tick {t} {key}")
        assert ra["vad_final"] == rb["vad_final"]


@pytest.mark.gpu
def test_errors_change_nothing(af):
    """No VAD, a stream index out of range and null arrays are refused (AF_ERR_INVALID) by the library itself, and the
    next push equals one without the call."""
    from audioflow import synth
    L = af.load_library()
    S, tick = 4, 960
    u32p, cp = C.POINTER(C.c_uint32), C.POINTER(af._VadConfigC)
    cfg = (af._VadConfigC * 2)(af.VadConfig(threshold_db=-20.0)._c(), af.VadConfig(smoothing_factor=0.05)._c())
    ids = (C.c_uint32 * 2)(1, S)
    novad = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False))
    s0 = af.Session(novad, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    assert L.af_session_set_vad_configs(s0._h, ids, cfg, 1) == af.AF_ERR_INVALID
    x = synth.stream(1, 0.5, 48000, 1)
    b0 = af.Batch(novad, [(x.ctypes.data, x.size, 48000, 1, af.AF_FMT_F32)], af.AF_MEM_HOST)
    assert L.af_batch_set_vad_configs(b0._h, cfg) == af.AF_ERR_INVALID
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    xs = [synth.stream(40 + i, 2.0, 48000, 1) for i in range(S)]
    for t in range(8):
        if t == 2:
            assert L.af_session_set_vad_configs(a._h, ids, cfg, 2) == af.AF_ERR_INVALID      # index S out of range
            assert L.af_session_set_vad_configs(a._h, None, cfg, 1) == af.AF_ERR_INVALID
            assert L.af_session_set_vad_configs(a._h, ids, C.cast(None, cp), 1) == af.AF_ERR_INVALID
            assert L.af_session_set_vad_configs(a._h, C.cast(None, u32p), None, 0) == af.AF_OK
        x = np.stack([xx[t * tick:(t + 1) * tick] for xx in xs])
        ra, rb = a.push(x), b.push(x)
        for key in ("pcm", "logmel", "vad"):
            assert_bit_equal(ra[key], rb[key], f"tick {t} {key}")
        assert ra["vad_final"] == rb["vad_final"]


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_config_replacement_keeps_the_state(orc):
    """_set_config on a hand-worked energy sequence: the state machine carries on under the new configuration."""
    c = orc.default_vad_config()
    c.smoothing_factor, c.threshold_db, c.silence_timeout_frames, c.min_speech_frames = 1.0, -50.0, 15, 3
    d = orc.VoiceActivityDetector(c)
    loud, quiet = 1e-2, 1e-8                                          # -40 dB and -160 dB (20 log10 of the energy)
    assert [d.detect_energy(e) for e in (quiet, loud, loud, loud, quiet, quiet, quiet)] == [0, 1, 1, 1, 1, 1, 1]
    assert (d.state(), d.silence_frames(), d.speech_frame_count()) == (SPEECH, 3, 3)
    c2 = orc.default_vad_config()
    c2.smoothing_factor, c2.threshold_db, c2.silence_timeout_frames, c2.min_speech_frames = 1.0, -50.0, 2, 3
    _set_config(d, c2)                                                  # timeout 2 below the silence count 3
    assert (d.state(), d.silence_frames(), d.speech_frame_count()) == (SPEECH, 3, 3)
    assert d.detect_energy(quiet) == 2                                # 4 >= 2, speech_frames 3 >= 3: Ending
    assert d.detect_energy(quiet) == 0
    c2.min_speech_frames = 5
    _set_config(d, c2)
    assert [d.detect_energy(e) for e in (loud, loud, quiet, quiet)] == [1, 1, 1, 0]    # 2 < 5 speech frames: no Ending
    c2.threshold_db = -10.0
    _set_config(d, c2)
    assert d.detect_energy(loud) == 0                                 # -40 dB is no longer speech


class _Cfg:
    def __init__(self, **kw):
        self.__dict__.update(kw)


def _stub(af, cls, n, vad=True):
    o = cls.__new__(cls)
    o._h = None
    o.pipe = _Cfg(cfg=_Cfg(vad_enable=int(vad)))
    if cls is af.Session:
        o.S = n
    else:
        o.n, o._owned = n, False
    return o


def test_python_argument_checks():
    """Batch.set_vad_configs / Session.set_vad_configs refuse bad arguments before calling the library."""
    import audioflow as af
    V = af.VadConfig
    s = _stub(af, af.Session, 4)
    with pytest.raises(ValueError, match="out of range"):
        s.set_vad_configs([4], [V()])
    with pytest.raises(ValueError, match="out of range"):
        s.set_vad_configs([-1], [V()])
    with pytest.raises(ValueError, match="2 streams and 1 configs"):
        s.set_vad_configs([0, 1], [V()])
    with pytest.raises(ValueError, match="not a VadConfig"):
        s.set_vad_configs([0], [dict(threshold_db=-40.0)])
    with pytest.raises(ValueError, match="silence_timeout_frames"):
        s.set_vad_configs([0], [V(silence_timeout_frames=-1)])
    with pytest.raises(ValueError, match="min_speech_frames"):
        s.set_vad_configs([0], [V(min_speech_frames=1 << 64)])
    with pytest.raises(ValueError, match="no VAD"):
        _stub(af, af.Session, 4, vad=False).set_vad_configs([0], [V()])
    b = _stub(af, af.Batch, 3)
    with pytest.raises(ValueError, match="2 configs for 3 streams"):
        b.set_vad_configs([V(), V()])
    with pytest.raises(ValueError, match="not a VadConfig"):
        b.set_vad_configs([V(), V(), None])
    with pytest.raises(ValueError, match="no VAD"):
        _stub(af, af.Batch, 3, vad=False).set_vad_configs(None)
