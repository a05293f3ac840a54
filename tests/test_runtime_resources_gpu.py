"""Every device and pinned allocation of the library is owned by one type that counts the live ones
(af_debug_live_allocations).  Each kind of handle -- sessions of one format and of mixed formats, with wire output,
levels, per-stream ticks and ring pushes; device and host batches; a one-rank sharded batch; a VAD object -- must raise
the counts while it lives and bring them back to where they stood once it is destroyed.  Unlike cudaMemGetInfo, the
counts see nothing of the other processes on the GPU."""
import ctypes as C
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _counts(af):
    gc.collect()
    return af.live_allocations()


def _noise(rng, shape, dtype=np.float32):
    return rng.normal(0.0, 0.05, shape).astype(dtype)


@pytest.fixture(scope="module")
def pipes(af):
    return {"mel": af.Pipeline(af.pipeline_config(n_mels=80)),
            "pcm16": af.Pipeline(af.pipeline_config(n_mels=80, pcm16=True))}


def _single_format_session(af, pipes, rng):
    s = af.Session(pipes["mel"], 8, 48000, 1, max_tick_samples=960)
    for _ in range(3):
        s.push(_noise(rng, (8, 960)))
    return s


def _mixed_format_session(af, pipes, rng):
    formats = [(48000, 1, 960), (44100, 1, 882), (16000, 2, 640)]
    s = af.Session.formats(pipes["mel"], formats, [0, 1, 2, 1, 0, 2])
    for t in range(4):
        xs = [_noise(rng, formats[f][2] - (t * 32 * formats[f][1] if k % 2 else 0)) for k, f in enumerate(s.stream_format)]
        s.push_streams(xs, end=[t == 1, 0, 0, 0, 0, t == 2])
        if t == 2:
            s.restart_streams([1, 2], [2, 0])
    return s


def _wire_session(af, pipes, rng):
    s = af.Session(pipes["mel"], 4, 48000, 1, max_tick_samples=960)
    plan = [(True, af.AF_MEM_HOST), (False, af.AF_MEM_DEVICE), (None, None), (True, af.AF_MEM_DEVICE),
            (False, af.AF_MEM_HOST), (None, None), (True, af.AF_MEM_HOST)]
    for gate, mem in plan:
        s.enable_wire(gate, mem=mem)
        s.push(_noise(rng, (4, 960)))
        if gate is not None:
            s.wire()
    return s


def _levels_session(af, pipes, rng):
    s = af.Session(pipes["mel"], 4, 44100, 1, max_tick_samples=882)
    for on in (True, False, True, True, False):
        s.enable_levels(on)
        s.push(_noise(rng, (4, 882)))
        if on:
            s.levels()
    return s


def _lazy_buffers_session(af, pipes, rng):
    """Host-mode per-stream ticks of a 44.1 kHz session (tick plan, fraction slices, PCM / log-mel / state staging) and
    both ring pushes (pinned staging rows)."""
    S = 6
    s = af.Session(pipes["mel"], S, 44100, 1, max_tick_samples=882)
    rings = [af.RingBuffer(8192) for _ in range(S)]
    s.push(_noise(rng, (S, 882)))
    s.push_streams([_noise(rng, 882 - 100 * k) for k in range(S)], end=[0, 1, 0, 0, 0, 0])
    for k, r in enumerate(rings):
        r.write(_noise(rng, 2000 + 50 * k))
    s.push_rings(rings, 441)
    s.push_rings_available(rings, 882)
    return s, rings


def _device_batch(af, pipes, pipe, rng):
    import torch
    from audioflow import synth
    x = synth.torch_batch(6, 2.0, 48000, 1, torch.device("cuda"), seed=5)
    b = pipes[pipe].batch([(x[i].data_ptr(), x.shape[1], 48000, 1, af.AF_FMT_F32) for i in range(6)], af.AF_MEM_DEVICE)
    pcm = torch.zeros((6, b.pcm_stride), device="cuda", dtype=torch.int16 if pipe == "pcm16" else torch.float32)
    lm = torch.zeros((6, b.logmel_stride), device="cuda")
    vad = torch.zeros((6, b.vad_stride), device="cuda", dtype=torch.uint8)
    torch.cuda.synchronize()
    # no energy rows (and i16 PCM rows with pcm16): the batch keeps its own scratch for them
    b.run_device(af.Batch.outputs_struct(pcm=pcm.data_ptr(), pcm_stride=b.pcm_stride, logmel=lm.data_ptr(),
                                         logmel_stride=b.logmel_stride, vad=vad.data_ptr(), vad_stride=b.vad_stride))
    torch.cuda.synchronize()
    return b, x, pcm, lm, vad


def _host_batch(af, pipes, streams):
    arrays = [x for x, _ in streams]
    b = pipes["mel"].batch([(x.ctypes.data, x.size, rate, 1, af.AF_FMT_F32) for x, rate in streams], af.AF_MEM_HOST)
    b.run_host(b.alloc_host_outputs())
    return b, arrays


def _host_batch_small(af, pipes, rng):
    return _host_batch(af, pipes, [(_noise(rng, 96000 + 441 * k), 48000 if k % 2 else 44100) for k in range(5)])


def _host_batch_many_subs(af, pipes, rng):
    """About 50 MB of input: two sub-batches of ~32 MB cycling through two slots.  The 170 s stream has more than 16384
    VAD frames, so its sub-batch also takes the scratch of the many-CTA scan."""
    streams = [(_noise(rng, 170 * 16000), 16000)] + [(_noise(rng, 40 * 48000), 48000) for _ in range(5)]
    return _host_batch(af, pipes, streams)


def _sharded_batch(af, pipes, rng):
    import torch
    from audioflow import synth
    x = synth.torch_batch(4, 2.0, 48000, 1, torch.device("cuda"), seed=6)
    sb = af.ShardedBatch(pipes["mel"], [(x[i].data_ptr(), x.shape[1], 48000, 1, af.AF_FMT_F32) for i in range(4)],
                         af.AF_MEM_DEVICE)
    b = sb.local(0)
    pcm = torch.zeros((4, b.pcm_stride), device="cuda")
    lm = torch.zeros((4, b.logmel_stride), device="cuda")
    torch.cuda.synchronize()
    outs = af.ShardedOutputsC()
    outs.shard[0] = af.Batch.outputs_struct(pcm=pcm.data_ptr(), pcm_stride=b.pcm_stride, logmel=lm.data_ptr(),
                                            logmel_stride=b.logmel_stride)
    sb.run(outs, gather=True)
    sb.gathered_host(0)
    return sb, x, pcm, lm


def _vad(af, pipes, rng):
    v = af.VoiceActivityDetector()
    v.detect_frames(_noise(rng, 16000), 400, 160)
    return v


# (builder, whether the object holds pinned host memory too)
CASES = {
    "session_single_format": (_single_format_session, False),
    "session_mixed_formats": (_mixed_format_session, True),
    "session_wire": (_wire_session, True),
    "session_levels": (_levels_session, True),
    "session_lazy_buffers": (_lazy_buffers_session, True),
    "batch_device": (lambda af, p, rng: _device_batch(af, p, "mel", rng), False),
    "batch_device_pcm16": (lambda af, p, rng: _device_batch(af, p, "pcm16", rng), False),
    "batch_host": (_host_batch_small, False),
    "batch_host_many_subs": (_host_batch_many_subs, False),
    "sharded_batch_one_rank": (_sharded_batch, False),
    "vad": (_vad, False),
}


@pytest.mark.parametrize("case", list(CASES))
def test_destroy_returns_every_allocation(af, pipes, case):
    build, pinned = CASES[case]
    try:
        # the first round fills what the process keeps across handles (the rate tables of 44.1 kHz batches, the
        # context's scratch); the second must end where it began
        for seed in (0, 1):
            before = _counts(af)
            obj = build(af, pipes, np.random.default_rng(seed))
            alive = _counts(af)
            assert alive[0] > before[0], (case, before, alive)
            if pinned:
                assert alive[1] > before[1], (case, before, alive)
            del obj
        assert _counts(af) == before, case
    finally:
        if case.startswith("sharded"):
            af.comm_shutdown()


def test_repeated_enables_allocate_nothing_more(af, pipes):
    rng = np.random.default_rng(7)
    s = af.Session(pipes["mel"], 4, 48000, 1, max_tick_samples=960)
    x = _noise(rng, (4, 960))
    s.push(x)
    s.enable_wire(True, mem=af.AF_MEM_HOST)
    s.enable_levels(True)
    s.push(x)
    first = _counts(af)
    for _ in range(4):
        s.enable_wire(True, mem=af.AF_MEM_HOST)
        s.enable_levels(False)
        s.enable_levels(True)
        s.push(x)
        s.wire()
        s.levels()
        assert _counts(af) == first
    s.enable_wire(None)
    off = _counts(af)
    assert off[0] < first[0] and off[1] < first[1]
    s.enable_wire(True, mem=af.AF_MEM_HOST)
    assert _counts(af) == first
    del s
    assert _counts(af)[0] < first[0]


def test_host_alloc_is_counted_until_freed(af):
    L = af.load_library()
    before = _counts(af)
    p = C.c_void_p()
    af._check(L.af_host_alloc(C.byref(p), 1 << 20))
    assert _counts(af) == (before[0], before[1] + 1)
    af._check(L.af_host_free(p))
    assert _counts(af) == before
