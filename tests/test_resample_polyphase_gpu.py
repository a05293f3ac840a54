"""Polyphase resampling of batches (af_batch_set_resampler(b, AF_RESAMPLE_POLYPHASE)): scipy.signal.resample_poly's
default anti-alias filter in place of the reference's cubic.  The taps are pinned to scipy's, the oracle's FIR
(orc_resample_polyphase, oracle/polyphase.c) to scipy's resample_poly, and the GPU's PCM to the oracle bit for bit.
Everything downstream must be what the batch computes for 16 kHz mono f32 rows holding that PCM; counts and strides must
not move."""
import ctypes as C

import numpy as np
import polyphase
import pytest

from test_parity_gpu import assert_bit_equal

RATES = [8000, 11025, 16000, 22050, 24000, 32000, 44100, 48000, 96000, 192000]
GPU_RATES = RATES + [88200]
# input frames: empty, one, under a 400-sample frame, and around the 48 kHz tile (1792 outputs) and the other ratios'
# tiles (up to 4096 outputs)
LENGTHS = [0, 1, 7, 399, 1199, 3 * 1792, 3 * 1792 + 1, 3 * 3584 + 2, 12287, 12290, 24577]


def _noise(seed, n_frames, ch, fmt):
    rng = np.random.default_rng(seed)
    if fmt == "i16":
        return rng.integers(-32768, 32768, n_frames * ch).astype(np.int16)
    return (0.5 * rng.standard_normal(n_frames * ch)).clip(-1, 1).astype(np.float32)


def _mono(orc, x, ch):
    return orc.to_mono(orc.i16_to_f32(x) if x.dtype == np.int16 else x, ch)


def _response_db(h, q, rate, freqs):
    """|H| in dB of the filter running at the upsampled rate rate * q (its DC gain is q)."""
    h = h.astype(np.float64) / q
    w = 2 * np.pi * np.asarray(freqs, np.float64) / (rate * q)
    i = np.arange(len(h))
    H = np.array([np.abs(np.dot(h, np.exp(-1j * wk * i))) for wk in w])
    return 20 * np.log10(np.maximum(H, 1e-300))


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def test_taps_are_scipys():
    import audioflow as af
    from scipy.signal import firwin
    report = []
    for rate in RATES:
        h, p, q = af.debug_polyphase_filter(rate)
        m = max(p, q)
        assert len(h) == 20 * m + 1
        if p == q == 1:                       # 16 kHz is copied; firwin has no filter at cutoff 1
            continue
        ref = firwin(20 * m + 1, 1.0 / m, window=("kaiser", 5.0)).astype(np.float32)
        ref *= q
        ulps = np.abs(h.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
        assert ulps.max() <= 1, (rate, int(ulps.max()))
        report.append((rate, int((ulps > 0).sum())))
    print("taps differing by 1 ulp:", report)


@pytest.mark.parametrize("rate", [r for r in RATES if r != 16000])
def test_filter_response(rate):
    import audioflow as af
    h, p, q = af.debug_polyphase_filter(rate)
    nyq = min(rate, 16000) / 2
    top = rate * q / 2
    pass_db = _response_db(h, q, rate, np.linspace(0, 0.75 * nyq, 200))
    assert np.abs(pass_db).max() <= 0.05, (rate, np.abs(pass_db).max())
    stop = np.concatenate([np.linspace(1.25 * nyq, min(top, 4 * nyq), 600), np.linspace(1.25 * nyq, top, 600)])
    stop_db = _response_db(h, q, rate, stop)
    assert stop_db.max() <= -55.0, (rate, stop_db.max())


@pytest.mark.parametrize("rate", [r for r in RATES if r != 16000])
def test_oracle_matches_resample_poly(orc, rate):
    import audioflow as af
    from scipy.signal import resample_poly
    h, p, q = af.debug_polyphase_filter(rate)
    m = _noise(rate, rate, 1, "f32")
    n_out = len(orc.resample_stream(m, rate, 16000))          # the cubic path's count, which the filter keeps
    y = polyphase.resample_polyphase(m, p, q, h, n_out)
    pad = np.zeros(n_out * p // q + 2 * p + 1, np.float32)    # zeros past the end, so scipy yields n_out outputs
    ref = resample_poly(np.concatenate([m, pad]), q, p)[:n_out].astype(np.float64)
    assert len(ref) == n_out
    err = np.abs(y.astype(np.float64) - ref)
    assert err.max() <= 1e-6, err.max()
    assert np.sqrt((err ** 2).sum() / (ref ** 2).sum()) <= 1e-6


def test_rate_outside_the_bound_has_no_filter():
    import audioflow as af
    L = af.load_library()
    p, q = C.c_uint32(0), C.c_uint32(0)
    assert L.af_debug_polyphase_filter(65537, 16000, None, 0, C.byref(p), C.byref(q)) == 0
    assert (p.value, q.value) == (65537, 16000)
    with pytest.raises(ValueError):
        af.debug_polyphase_filter(65537)


def test_unknown_filter_name_is_refused_before_the_library(monkeypatch):
    import audioflow as af
    b = af.Batch.__new__(af.Batch)
    b._h, b._owned = None, False

    def no_library():
        raise AssertionError("the library was called")
    monkeypatch.setattr(af, "load_library", no_library)
    for name in ("sinc", "Polyphase", "", "linear"):
        with pytest.raises(ValueError):
            b.set_resampler(name)
    sb = af.ShardedBatch.__new__(af.ShardedBatch)
    sb._h, sb.n_ranks = None, 1
    with pytest.raises(ValueError):
        sb.set_resampler("kaiser")


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _desc(af, x, ptr, rate, ch):
    return (ptr, x.size, rate, ch, af.AF_FMT_I16 if x.dtype == np.int16 else af.AF_FMT_F32)


def _run_host(af, pipe, streams, filt=None):
    b = af.Batch(pipe, [_desc(af, x, x.ctypes.data, r, ch) for x, r, ch in streams], af.AF_MEM_HOST)
    if filt:
        b.set_resampler(filt)
    out = b.alloc_host_outputs()
    b.run_host(out)
    return b, b.split(out)


def _run_device(af, pipe, streams, filt=None, cfgs=None, rows=None):
    """A device batch: streams as (x, rate, ch) host arrays copied to the GPU, or rows=(tensor, n per row) of 16 kHz f32
    device rows.  Returns (batch, per-stream results)."""
    import torch
    dev = torch.device("cuda")
    if rows is None:
        keep = [torch.from_numpy(x.copy()).to(dev) for x, _, _ in streams]
        descs = [_desc(af, x, t.data_ptr(), r, ch) for (x, r, ch), t in zip(streams, keep)]
    else:
        t, ns = rows
        keep = [t]
        descs = [(t[i].data_ptr(), int(n), 16000, 1, af.AF_FMT_F32) for i, n in enumerate(ns)]
    b = af.Batch(pipe, descs, af.AF_MEM_DEVICE)
    if filt:
        b.set_resampler(filt)
    if cfgs is not None:
        b.set_vad_configs(cfgs)
    cfg, S = pipe.cfg, max(len(descs), 1)
    pcm = torch.zeros((S, b.pcm_stride), device=dev, dtype=torch.int16 if cfg.pcm16 else torch.float32)
    lm = torch.zeros((S, b.logmel_stride), device=dev)
    vad = torch.zeros((S, b.vad_stride), device=dev, dtype=torch.uint8)
    en = torch.zeros((S, b.energy_stride), device=dev)
    fin = torch.zeros((S, 6), device=dev, dtype=torch.int32)
    o = af.OutputsC(pcm.data_ptr(), b.pcm_stride, lm.data_ptr() if cfg.n_mels else None, b.logmel_stride,
                    vad.data_ptr() if cfg.vad_enable else None, b.vad_stride,
                    en.data_ptr() if cfg.vad_enable else None, b.energy_stride,
                    fin.data_ptr() if cfg.vad_enable else None)
    torch.cuda.synchronize()
    b.run_device(o)
    torch.cuda.synchronize()
    res = []
    M = cfg.n_mels
    for i in range(len(descs)):
        n, T, V = int(b.n_out[i]), int(b.n_feat[i]), int(b.n_vad[i])
        res.append({"pcm": pcm[i, :n].cpu().numpy() if cfg.write_pcm else None,
                    "logmel": lm[i, :T * M].cpu().numpy() if M else None,
                    "vad": vad[i, :V].cpu().numpy() if cfg.vad_enable else None,
                    "energy": en[i, :V].cpu().numpy() if cfg.vad_enable else None,
                    "vad_final": fin[i].cpu().numpy() if cfg.vad_enable else None})
    res_rows = pcm if not cfg.pcm16 else None
    return b, res, res_rows, keep


def _oracle_pcm(af, orc, x, rate, ch, n_out):
    h, p, q = af.debug_polyphase_filter(rate)
    return polyphase.resample_polyphase(_mono(orc, x, ch), p, q, h, n_out)


def _formats_streams(rate):
    out = []
    for ch in (1, 2, 6):
        for fmt in ("f32", "i16"):
            for k, n in enumerate(LENGTHS):
                out.append((_noise(rate + 97 * ch + 13 * k + (fmt == "i16"), n, ch, fmt), rate, ch))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("rate", GPU_RATES)
def test_pcm_matches_oracle(af, orc, rate):
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False))
    streams = _formats_streams(rate)
    bh, host = _run_host(af, pipe, streams, "polyphase")
    bd, dev, _, _ = _run_device(af, pipe, streams, "polyphase")
    for i, (x, r, ch) in enumerate(streams):
        ref = _oracle_pcm(af, orc, x, r, ch, int(bh.n_out[i]))
        what = f"{rate} Hz, {ch} ch, {x.dtype}, {x.size // ch} frames"
        assert_bit_equal(host[i]["pcm"], ref, "host " + what)
        assert_bit_equal(dev[i]["pcm"], ref, "device " + what)


@pytest.mark.gpu
def test_mixed_rate_batch(af, orc):
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False))
    streams = [(_noise(5 + i, 4000 + 977 * i, 1 + i % 3, "i16" if i % 4 == 3 else "f32"), r, 1 + i % 3)
               for i, r in enumerate(GPU_RATES * 2)]
    bh, host = _run_host(af, pipe, streams, "polyphase")
    _, dev, _, _ = _run_device(af, pipe, streams, "polyphase")
    for i, (x, r, ch) in enumerate(streams):
        ref = _oracle_pcm(af, orc, x, r, ch, int(bh.n_out[i]))
        assert_bit_equal(host[i]["pcm"], ref, f"host stream {i} ({r} Hz)")
        assert_bit_equal(dev[i]["pcm"], ref, f"device stream {i} ({r} Hz)")


@pytest.mark.gpu
def test_cfg4_hour_48k_stereo(af, orc):
    from audioflow import synth
    x = synth.stream(4, 3600.0, 48000, 2)
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False))
    b, dev, _, keep = _run_device(af, pipe, [(x, 48000, 2)], "polyphase")
    del keep
    ref = _oracle_pcm(af, orc, x, 48000, 2, int(b.n_out[0]))
    assert_bit_equal(dev[0]["pcm"], ref, "one hour, 48 kHz stereo")


def _same(g, r, what):
    for k in ("pcm", "logmel", "vad", "energy", "vad_final"):
        if r[k] is not None or g[k] is not None:
            assert_bit_equal(g[k], r[k], f"{what}: {k}")


DOWNSTREAM = {
    "default": dict(n_mels=80),
    "pcm16": dict(n_mels=80, pcm16=True),
    "no_pcm": dict(n_mels=80, write_pcm=False),
    "vad_320": dict(n_mels=128, vad_frame_len=320, vad_hop=320),
    "vad_configs": dict(n_mels=80),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(DOWNSTREAM))
def test_downstream_is_that_of_16k_rows(af, orc, case):
    """Log-mel, energies, states and vad_final of a polyphase batch are those of a cubic batch over 16 kHz f32 device
    rows holding the polyphase PCM."""
    import torch
    from audioflow import synth
    streams = [(synth.stream(40 + i, 0.7 + 0.9 * i, r, ch), r, ch)
               for i, (r, ch) in enumerate([(48000, 1), (44100, 2), (48000, 2), (22050, 1), (96000, 6), (8000, 1)])]
    streams.append((np.zeros(0, np.float32), 48000, 1))
    cfgs = None
    if case == "vad_configs":
        V = af.VadConfig
        cfgs = [V(), V(threshold_db=-35.0), V(smoothing_factor=0.05), V(silence_timeout_frames=1), V(min_speech_frames=10),
                V(-60.0, 0.1, 5, 1), V()]
    plain = af.Pipeline(af.pipeline_config(n_mels=80))
    bp, src, rows, keep = _run_device(af, plain, streams, "polyphase")            # the polyphase PCM as f32 rows
    pipe = af.Pipeline(af.pipeline_config(**DOWNSTREAM[case]))
    b, got, _, _ = _run_device(af, pipe, streams, "polyphase", cfgs)
    ref_rows = rows.clone()
    br, ref, _, _ = _run_device(af, pipe, None, None, cfgs, rows=(ref_rows, bp.n_out[:len(streams)]))
    assert np.array_equal(b.n_out, br.n_out) and np.array_equal(b.n_feat, br.n_feat) and np.array_equal(b.n_vad, br.n_vad)
    for i in range(len(streams)):
        _same(got[i], ref[i], f"{case}, stream {i}")
    for i, (x, r, ch) in enumerate(streams):                 # the rows themselves are the oracle's
        assert_bit_equal(src[i]["pcm"], _oracle_pcm(af, orc, x, r, ch, int(bp.n_out[i])), f"stream {i} pcm")
    del keep
    torch.cuda.synchronize()


def _counts(af, b):
    L = af.load_library()
    n = max(b.n, 1)
    no, nf, nv = (np.zeros(n, np.uint32) for _ in range(3))
    u32p = C.POINTER(C.c_uint32)
    af._check(L.af_batch_counts(b._h, no.ctypes.data_as(u32p), nf.ctypes.data_as(u32p), nv.ctypes.data_as(u32p)))
    ps, ls, vs = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
    af._check(L.af_batch_strides(b._h, C.byref(ps), C.byref(ls), C.byref(vs)))
    return no.tolist(), nf.tolist(), nv.tolist(), (ps.value, ls.value, vs.value)


@pytest.mark.gpu
def test_counts_strides_and_switching_back(af):
    from audioflow import synth
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    streams = [(synth.stream(60 + i, 1.3 + i, r, 1), r, 1) for i, r in enumerate([48000, 44100, 16000, 11025])]
    descs = [_desc(af, x, x.ctypes.data, r, ch) for x, r, ch in streams]
    b = af.Batch(pipe, descs, af.AF_MEM_HOST)
    before = _counts(af, b)
    a0 = af.live_allocations()
    out = b.alloc_host_outputs()
    b.run_host(out)
    cubic = b.split(out)
    l0 = af.kernel_launch_count()
    b.set_resampler("polyphase")
    assert _counts(af, b) == before
    assert af.live_allocations()[0] > a0[0]
    out = b.alloc_host_outputs()
    b.run_host(out)
    poly = b.split(out)
    assert not np.array_equal(poly[0]["pcm"], cubic[0]["pcm"])
    b.set_resampler("cubic")
    assert _counts(af, b) == before
    assert af.live_allocations() == a0
    out = b.alloc_host_outputs()
    l1 = af.kernel_launch_count()
    b.run_host(out)
    launches = af.kernel_launch_count() - l1
    for i, (g, r) in enumerate(zip(b.split(out), cubic)):
        _same(g, r, f"cubic again, stream {i}")
    b.set_resampler("polyphase")                            # one more FIR launch per sub-batch than the cubic run
    out = b.alloc_host_outputs()
    l2 = af.kernel_launch_count()
    b.run_host(out)
    assert af.kernel_launch_count() - l2 == launches + 1
    for i, (g, r) in enumerate(zip(b.split(out), poly)):
        _same(g, r, f"polyphase again, stream {i}")
    del b
    assert l0 <= af.kernel_launch_count()


@pytest.mark.gpu
def test_refused_rate_keeps_the_previous_filter(af):
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    streams = [(_noise(1, 48000, 1, "f32"), 48000, 1), (_noise(2, 65537, 1, "f32"), 65537, 1)]
    b, cubic = _run_host(af, pipe, streams)
    a0 = af.live_allocations()
    L = af.load_library()
    assert L.af_batch_set_resampler(b._h, 1) == af.AF_ERR_RESAMPLING_FAILED
    assert "stream 1" in af.last_error()
    assert L.af_batch_set_resampler(b._h, 2) == af.AF_ERR_INVALID
    assert L.af_batch_set_resampler(None, 1) == af.AF_ERR_INVALID
    assert af.live_allocations() == a0
    out = b.alloc_host_outputs()
    b.run_host(out)
    for i, (g, r) in enumerate(zip(b.split(out), cubic)):
        _same(g, r, f"after the refusal, stream {i}")


def _tone(rate, f, seconds=1.0, amp=0.5):
    t = np.arange(int(seconds * rate)) / rate
    return (amp * np.sin(2 * np.pi * f * t)).astype(np.float32)


def _rms_db(y, x):
    return 20 * np.log10(np.sqrt(np.mean(y.astype(np.float64) ** 2)) / np.sqrt(np.mean(x.astype(np.float64) ** 2)))


@pytest.mark.gpu
def test_aliasing(af):
    pipe = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False))
    cases = [(48000, 12000.0), (44100, 11000.0), (48000, 1000.0)]
    streams = [(_tone(r, f), r, 1) for r, f in cases]
    _, cubic = _run_host(af, pipe, streams)
    _, poly = _run_host(af, pipe, streams, "polyphase")
    for (r, f), (x, _, _), c, p in zip(cases, streams, cubic, poly):
        cut = slice(200, -200)                          # away from the filter's start-up at the stream edges
        dp, dc = _rms_db(p["pcm"][cut], x), _rms_db(c["pcm"][cut], x)
        print(f"{f:.0f} Hz at {r} Hz: polyphase {dp:.2f} dB, cubic {dc:.2f} dB")
        if f > 8000:
            assert dp <= -60.0, (r, f, dp)
            assert dc >= -3.0, (r, f, dc)               # the cubic path folds it into the speech band
        else:
            assert abs(dp) <= 0.05, (r, f, dp)


def _n_gpus():
    import audioflow
    n = C.c_int(0)
    try:
        audioflow.load_library().af_device_count(C.byref(n))
    except Exception:
        return 0
    return n.value


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs 2 GPUs")
def test_sharded_polyphase_matches_one_gpu(af, orc):
    import torch
    streams = [(_noise(70 + i, 20000 + 3331 * i, 1, "f32"), 44100 if i % 2 else 48000, 1) for i in range(10)]
    af.init_multi(2)
    try:
        geo = [(0, x.size, r, 1, af.AF_FMT_F32) for x, r, _ in streams]
        parts = af.shard_partition(geo, 2)
        owner = [0 if i < parts[0][1] else 1 for i in range(len(streams))]
        dx = [torch.tensor(x, device=f"cuda:{owner[i]}") for i, (x, _, _) in enumerate(streams)]
        descs = [(dx[i].data_ptr(), x.size, r, 1, af.AF_FMT_F32) for i, (x, r, _) in enumerate(streams)]
        pipe = af.Pipeline(af.pipeline_config(n_mels=80))
        sb = af.ShardedBatch(pipe, descs, af.AF_MEM_DEVICE)
        sb.set_resampler("polyphase")
        outs = af.ShardedOutputsC()
        bufs = []
        for r in range(2):
            lo, cnt, dev = sb.shard(r)
            b = sb.local(r)
            d = torch.device("cuda", r)
            pcm = torch.zeros((cnt, b.pcm_stride), device=d)
            lm = torch.zeros((cnt, b.logmel_stride), device=d)
            outs.shard[r] = af.OutputsC(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, None, 0, None, 0, None)
            bufs.append((lo, cnt, b, pcm, lm))
        for d in range(2):
            torch.cuda.synchronize(d)
        sb.run(outs, gather=True, wait=True)
        for d in range(2):
            torch.cuda.synchronize(d)
        got = {}
        for lo, cnt, b, pcm, lm in bufs:
            for li in range(cnt):
                got[lo + li] = (pcm[li, :int(b.n_out[li])].cpu().numpy(), lm[li, :int(b.n_feat[li]) * 80].cpu().numpy())
        del sb
    finally:
        af.comm_shutdown()
        af.init(0)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    for i, s in enumerate(streams):
        b, one, _, _ = _run_device(af, pipe, [s], "polyphase")
        assert_bit_equal(got[i][0], one[0]["pcm"], f"stream {i} pcm")
        assert_bit_equal(got[i][1], one[0]["logmel"], f"stream {i} log-mel")
