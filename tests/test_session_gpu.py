"""GPU tests of the streaming sessions (BASELINE config 5): persistent per-stream state across ticks must
reproduce exactly what the reference objects produce when fed the same chunks:
BatchResampler::process per tick (resampler.rs:132-147), detect per completed frame (vad.rs:97-154)."""
import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal, assert_logmel_close

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("rate,tick,fmt,ch", [(48000, 960, "f32", 1), (44100, 882, "f32", 1), (48000, 1000, "i16", 2),
                                               (16000, 320, "f32", 1), (32000, 77, "f32", 1)])
def test_session_matches_reference_objects(af, orc, rate, tick, fmt, ch):
    from audioflow import synth
    S, n_ticks = 5, 40
    total = tick * n_ticks
    xs = [synth.stream(60 + i, total / rate + 0.01, rate, ch, fmt)[: total * ch] for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    ses = af.Session(pipe, S, rate, ch, af.AF_FMT_I16 if fmt == "i16" else af.AF_FMT_F32, max_tick_samples=tick * ch)
    pcm = [[] for _ in range(S)]
    lm = [[] for _ in range(S)]
    vad = [[] for _ in range(S)]
    per_tick_counts = []
    dets = [orc.VoiceActivityDetector() for _ in range(S)]
    carry = [np.zeros(0, np.float32) for _ in range(S)]
    for t in range(n_ticks):
        x = np.stack([xs[i][t * tick * ch:(t + 1) * tick * ch] for i in range(S)])
        r = ses.push(x)
        per_tick_counts.append(r["pcm"].shape[1])
        for i in range(S):
            pcm[i].append(r["pcm"][i]); lm[i].append(r["logmel"][i]); vad[i].append(r["vad"][i])
            # vad_final after every tick, frameless ones included: the detector fed the frames completed so far
            carry[i] = np.concatenate([carry[i], r["pcm"][i]])
            while len(carry[i]) >= 400:
                dets[i].detect(carry[i][:400])
                carry[i] = carry[i][160:]
            fin = r["vad_final"][i]
            assert (fin["state"], fin["speech_frames"]) == (dets[i].state(), dets[i].speech_frame_count()), (t, i)
            assert np.float32(fin["smoothed"]).view(np.uint32) == np.float32(dets[i].smoothed_energy()).view(np.uint32), (t, i)
    for i in range(S):
        xi = orc.i16_to_f32(xs[i]) if fmt == "i16" else xs[i]
        mono = orc.to_mono(xi, ch)
        b = orc.BatchResampler(rate, 16000)
        ref_chunks = [b.process(mono[t * tick:(t + 1) * tick]) for t in range(n_ticks)]
        if i == 0:
            assert per_tick_counts == [len(c) for c in ref_chunks]          # per-call output counts (chunk recurrence)
        ref_pcm = np.concatenate(ref_chunks)
        got_pcm = np.concatenate(pcm[i])
        assert_bit_equal(got_pcm, ref_pcm, f"session pcm {i}")
        T = orc.num_frames(len(ref_pcm))
        got_vad = np.concatenate(vad[i])
        got_lm = np.concatenate(lm[i])
        assert len(got_vad) == T and got_lm.shape == (T, 80)
        v = orc.VoiceActivityDetector()
        st, _ = v.stream(ref_pcm, 400, 160)
        assert_bit_equal(got_vad, st, f"session vad {i}")
        assert_logmel_close(got_lm, orc.logmel(ref_pcm, orc.default_feat_config(80)), f"session logmel {i}")
    fin = r["vad_final"][S - 1]
    assert fin["state"] == v.state() and fin["speech_frames"] == v.speech_frame_count()


def test_session_reset_and_20ms_vad(af, orc):
    """resample + VAD on 20 ms frames only (the reference's intended loop), two passes separated by reset()."""
    from audioflow import synth
    S, tick, n_ticks = 3, 960, 25
    xs = [synth.stream(80 + i, 0.6, 48000, 1)[: tick * n_ticks] for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad_frame_len=320, vad_hop=320))
    ses = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    for rep in range(2):
        vad = [[] for _ in range(S)]
        for t in range(n_ticks):
            r = ses.push(np.stack([x[t * tick:(t + 1) * tick] for x in xs]))
            for i in range(S):
                vad[i].append(r["vad"][i])
        for i in range(S):
            b = orc.BatchResampler(48000, 16000)
            ref_pcm = np.concatenate([b.process(xs[i][t * tick:(t + 1) * tick]) for t in range(n_ticks)])
            st, _ = orc.VoiceActivityDetector().stream(ref_pcm, 320, 320)
            assert_bit_equal(np.concatenate(vad[i]), st, f"rep {rep} stream {i}")
        ses.reset()


def test_session_fed_by_capture_rings(af, orc):
    """The capture hand-off (RingBuffer, capture.rs:84-161 -> AudioCapturer::read_frame, capture.rs:310-319): producer
    chunks of uneven size go into one ring per stream, ticks of 960 samples come out; the session must produce exactly
    what pushing the same samples directly produces, and a tick must consume nothing unless every ring can serve it."""
    from audioflow import synth
    S, tick, n_ticks, rate = 4, 960, 12, 48000
    xs = [synth.stream(90 + i, tick * n_ticks / rate + 0.01, rate, 1)[: tick * n_ticks] for i in range(S)]
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    direct = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    ringed = af.Session(pipe, S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    rings = [af.RingBuffer(4096) for _ in range(S)]
    fed = [0] * S
    rng = np.random.default_rng(5)
    for t in range(n_ticks):
        # cpal-style producer: irregular callback sizes until every ring holds a tick
        while min(r.available() for r in rings) < tick:
            for i in range(S):
                n = int(rng.integers(100, 700))
                n = min(n, len(xs[i]) - fed[i])
                fed[i] += rings[i].write(xs[i][fed[i]:fed[i] + n])
        a = direct.push(np.stack([xs[i][t * tick:(t + 1) * tick] for i in range(S)]))
        b = ringed.push_rings(rings, tick)
        for k in ("pcm", "logmel", "vad"):
            assert_bit_equal(a[k], b[k], f"tick {t} {k}")
    # a ring that cannot serve the tick: error, nothing consumed anywhere
    before = [r.available() for r in rings]
    rings[2].clear()
    before[2] = 0
    with pytest.raises(ValueError):                     # AF_ERR_INVALID
        ringed.push_rings(rings, tick)
    assert [r.available() for r in rings] == before


def test_session_levels(af, orc):
    """AudioLevel{level, peak} / VolumeLevel{level, is_speech} (events/mod.rs:41, modules/events/mod.rs:22) per tick:
    level = energy_db() and is_speech = is_speaking() of the reference detector fed the same frames (vad.rs:192-199),
    peak = max |y| of the tick's 16 kHz samples -- all three bit-exact."""
    from audioflow import synth
    S, tick, n_ticks, rate = 3, 960, 30, 48000
    xs = [synth.stream(120 + i, tick * n_ticks / rate + 0.01, rate, 1)[: tick * n_ticks] for i in range(S)]
    ses = af.Session(af.Pipeline(af.pipeline_config(n_mels=80)), S, rate, 1, af.AF_FMT_F32, max_tick_samples=tick)
    with pytest.raises(ValueError):
        ses.levels()                                              # not enabled / no tick yet
    ses.enable_levels()
    dets = [orc.VoiceActivityDetector() for _ in range(S)]
    carry = [np.zeros(0, np.float32) for _ in range(S)]
    for t in range(n_ticks):
        r = ses.push(np.stack([xs[i][t * tick:(t + 1) * tick] for i in range(S)]))
        lv = ses.levels()
        for i in range(S):
            y = r["pcm"][i]
            want_peak = np.float32(np.max(np.abs(y))) if len(y) else np.float32(0)
            assert lv["peak"][i].view(np.uint32) == want_peak.view(np.uint32)
            carry[i] = np.concatenate([carry[i], y])
            while len(carry[i]) >= 400:                           # the detector sees every completed 25 ms / 10 ms frame
                dets[i].detect(carry[i][:400])
                carry[i] = carry[i][160:]
            want_db = np.float32(dets[i].energy_db())
            got_db = lv["level_db"][i]
            assert (np.isneginf(want_db) and np.isneginf(got_db)) or got_db.view(np.uint32) == want_db.view(np.uint32), (t, i, got_db, want_db)
            assert bool(lv["is_speech"][i]) == dets[i].is_speaking()
