"""Every resampler path the batch planner can choose, against the oracle.

Three inputs of a stream select the code the fused kernel's resampler role runs: the rate (position mode: passthrough,
exact recurrence with q == 1 or q > 1, fraction table through the periodic-offset path or the plain rational path), the
channel count and the sample format (kind: mono / stereo in f32 / i16, or the checked-only generic kind for 3 and more
channels), and the bytes one part of a step needs (staging: two parts, four quarter parts, or not staged at all, with
unchecked taps straight from global memory).  Batch composition changes the code too: only the first table rate of a
batch gets the periodic path, and a batch with a quarter-staged stream runs every stream in the QUARTERS kernel instance.

The case matrix below spans those paths at lengths that end on the planner's edges (two tiles, two tiles + 1, a part
boundary inside a step, one sample before a step boundary).  test_matrix_spans_every_path (CPU) derives each case's path
from the library's own planning and the constants of af_common.cuh, so a change of the stage size cannot quietly empty a
row.  The GPU tests run every case alone, in one mixed batch under both kernel variants, and in that batch on device
buffers that start 16 bytes past a 256-byte boundary; PCM, frame energies, VAD states and the final detector state
bit-exact, log-mel within _assert_logmel.  The same rates go through the two other resampler implementations
(a one-stream Session and BatchResampler), which show what the fused kernel has to match."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from test_parity_gpu import LOGMEL_REL_L2, _check_stream, assert_bit_equal, logmel_tolerance
from test_session_streams_gpu import Harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMMON = os.path.join(ROOT, "audio-flow-rs_b200", "csrc", "af_common.cuh")
OUT_RATE = 16000
RS_PASSTHROUGH, RS_EXACT, RS_TABLE = 0, 1, 2


# ---------------------------------------------------------------------------------------------------------------------
# the planner's constants, read from the header so that a change to them is followed
# ---------------------------------------------------------------------------------------------------------------------
def _geometry():
    src = open(COMMON).read()
    ints = {}
    for name, v in re.findall(r"constexpr int (\w+) = (\d+);", src):
        ints.setdefault(name, int(v))        # (the first of two #ifdef branches: the warp counts sum the same)
    m = re.search(r"part_max_out\(int parts\)\s*\{\s*return parts == 4 \? (\d+) : (\d+);", src)
    assert m, "part_max_out not found in af_common.cuh"
    g = dict(STAGE_BYTES=ints["STAGE_BYTES"], KOFF_MAX=ints["KOFF_MAX"], PART_MAX={4: int(m.group(1)), 2: int(m.group(2))},
             HOP=ints["HOP"], WIN=ints["WIN"], SF=ints["SF"], TILE_FRAMES=ints["TILE_FRAMES"])
    g["STEP"] = g["SF"] * g["HOP"]
    g["TILE"] = g["TILE_FRAMES"] * g["HOP"]
    g["YLEN"] = g["STEP"] + g["WIN"] - g["HOP"]
    g["THREADS"] = 32 * (ints["FFT_WARPS"] + ints["MEL_WARPS"] + ints["VAD_WARPS"] + ints["RS_WARPS"])
    return g


GEO = _geometry()
TILE, STEP = GEO["TILE"], GEO["STEP"]


def _mode(rate):
    import audioflow
    m = C.c_int(-1)
    audioflow.load_library().af_debug_resample_plan(rate, OUT_RATE, 0, None, 0, C.byref(m))
    return m.value


def plan(rate, ch, fmt, n_out):
    """The path of one stream, as build_sub / plan_tile (af_runtime.cu, af_device.cuh) and the resampler role's dispatch
    (af_fused.cu) choose it."""
    g = math.gcd(rate, OUT_RATE)
    p, q = rate // g, OUT_RATE // g
    mode = _mode(rate)
    bps = 2 if fmt == "i16" else 4
    staged = 0
    for parts in (2, 4):
        outs = GEO["PART_MAX"][parts]
        frames = outs if mode == RS_PASSTHROUGH else -(-outs * p // q)
        if not staged and ch <= 2 and (frames + 8) * ch * bps + 32 <= GEO["STAGE_BYTES"]:
            staged = parts
    periodic = (mode == RS_TABLE and q <= GEO["KOFF_MAX"] and q % 4 == 0 and STEP % q == 0 and p < 65536)
    kind = "generic" if ch > 2 else f"{fmt}x{ch}"
    if mode == RS_PASSTHROUGH:
        pos = "passthrough"
    elif mode == RS_EXACT:
        pos = ("exact_48k" if p == 3 else "exact_q1") if q == 1 else "exact_rational"
    else:
        pos = "table_q1" if q == 1 else ("table_periodic" if periodic else "table_rational")
    return dict(rate=rate, p=p, q=q, mode=mode, kind=kind, staged=staged if kind != "generic" else 0, periodic=periodic,
                pos=pos, n_out=n_out, tiles=-(-n_out // TILE))


# ---------------------------------------------------------------------------------------------------------------------
# the case matrix
# ---------------------------------------------------------------------------------------------------------------------
RATES = [4000, 8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000, 49000, 64000, 88200, 96000, 96190, 96200,
         176400, 192000, 47999, 16001, 15999]
EXTREMES = [160001, 1888000, 784000, 1488000]     # largest accepted p; largest accepted step; two q == 1 table rates
KINDS = [(1, "f32"), (1, "i16"), (2, "f32"), (2, "i16")]
GENERIC = [(4, "f32", 48000), (6, "i16", 44100), (8, "f32", 16000), (4, "i16", 96000), (6, "f32", 22050),
           (8, "i16", 8000), (4, "f32", 11025), (8, "f32", 192000)]
TARGETS = ["2tiles", "2tiles+1", "part", "step-1"]


def _target(name, staged):
    return {"2tiles": 2 * TILE, "2tiles+1": 2 * TILE + 1, "step-1": 2 * TILE + STEP - 1,
            "part": 2 * TILE + GEO["PART_MAX"][4 if staged == 4 else 2]}[name]


def _n_in_for(rate, want, past):
    """n_in of a stream that ends on an edge of the planner: the largest whose output length does not pass `want`, or
    (past=True, one output past an edge) the smallest that reaches it.  Outputs grow one 128-frame chunk at a time, so
    below 16 kHz and at most rates above it the edge itself cannot be hit exactly."""
    import audioflow
    lo, hi = 1, 128 * (want * rate // OUT_RATE // 128 + 64)
    assert audioflow.resample_output_len(rate, OUT_RATE, hi) > want
    while lo < hi:                          # smallest n with len(n) >= want + (not past)
        mid = (lo + hi) // 2
        if audioflow.resample_output_len(rate, OUT_RATE, mid) >= want + (0 if past else 1):
            hi = mid
        else:
            lo = mid + 1
    return lo if past else lo - 1


def _cases():
    """(name, seed, rate, channels, fmt, target, drop): `drop` interleaved samples cut off the end (a trailing partial
    channel frame).  The first table rate is 11025 Hz (q = 640 = KOFF_MAX): in the mixed batch it keeps the periodic
    path and every other table rate, 44.1 kHz included, takes the plain rational one."""
    out = []
    for i, rate in enumerate(RATES):
        for j, (ch, fmt) in enumerate(KINDS):
            drop = 1 if (ch == 2 and (i + j) % 5 == 0) else 0
            out.append((f"{rate}-{fmt}x{ch}-{TARGETS[(i + j) % 4]}", 1000 + 4 * i + j, rate, ch, fmt, TARGETS[(i + j) % 4], drop))
    for i, (ch, fmt, rate) in enumerate(GENERIC):
        out.append((f"{rate}-{fmt}x{ch}-{TARGETS[i % 4]}", 1200 + i, rate, ch, fmt, TARGETS[i % 4], (i % ch) if i % 2 else 0))
    for i, rate in enumerate(EXTREMES):
        for j, (ch, fmt) in enumerate(KINDS):
            out.append((f"{rate}-{fmt}x{ch}-2tiles+1", 1300 + 4 * i + j, rate, ch, fmt, "2tiles+1", 1 if ch == 2 and j == 3 else 0))
    return out


CASES = _cases()
CASE_IDS = [c[0] for c in CASES]


def _geometry_of(case):
    """(n_in, n_out, plan) of a case (_n_in_for)."""
    import audioflow
    name, seed, rate, ch, fmt, target, drop = case
    staged = plan(rate, ch, fmt, 0)["staged"]
    n_in = _n_in_for(rate, _target(target, staged), target == "2tiles+1")
    n_out = audioflow.resample_output_len(rate, OUT_RATE, n_in)
    return n_in, n_out, plan(rate, ch, fmt, n_out)


def _signal(case):
    from audioflow import synth
    name, seed, rate, ch, fmt, target, drop = case
    n_in, _, _ = _geometry_of(case)
    x = synth.stream(seed, (n_in + 2) / rate, rate, ch, fmt)[:n_in * ch]
    assert len(x) == n_in * ch
    return x[:len(x) - drop] if drop else x


def _specials(case):
    """The signal of a case with the values that break shortcuts sprinkled in: +-0, runs of zeros, |x| >= 2, subnormals,
    +-Inf and NaN (f32); runs of -32768, 32767 and 0 (i16)."""
    x = _signal(case).copy()
    rng = np.random.default_rng(case[1] + 77)
    n = len(x)
    if x.dtype == np.int16:
        for k in range(400):
            x[int(rng.integers(0, n))] = (-32768, 32767, 0, 1, -1)[k % 5]
        for k in range(24):
            s = int(rng.integers(0, n - 400))
            x[s:s + int(rng.integers(3, 400))] = (-32768, 32767, 0)[k % 3]
        return x
    specials = np.array([0.0, -0.0, 2.0, -2.0, 1.9999999, 3.5, -7.25, 1e30, -1e30, 1e-40, -1e-41, 1.17549435e-38,
                         np.inf, -np.inf, np.nan, 65504.0, 1.0, -1.0], np.float32)
    for k in range(400):
        x[int(rng.integers(0, n))] = specials[k % len(specials)]
    for k in range(24):
        s = int(rng.integers(0, n - 400))
        x[s:s + int(rng.integers(3, 400))] = (0.0, -0.0, 2.5, 1e-39)[k % 4]
    return x


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the matrix spans every path (the review aid: what the GPU tests below cover, on any machine)
# ---------------------------------------------------------------------------------------------------------------------
def test_matrix_spans_every_path():
    P = []
    for case in CASES:
        n_in, n_out, pl = _geometry_of(case)
        name, seed, rate, ch, fmt, target, drop = case
        pl.update(name=name, target=target, n_in=n_in, nbytes=(n_in * ch - drop) * (2 if fmt == "i16" else 4), drop=drop, ch=ch,
                  fmt=fmt)
        P.append(pl)
    fast = [c for c in P if c["kind"] != "generic"]

    def some(what, pred):
        hit = [c["name"] for c in P if pred(c)]
        assert hit, f"no case takes the path: {what}"
        return hit

    # lengths: every target, by staging (quarter-staged streams end on their own part boundary)
    for t in TARGETS:
        for st in (2, 4, 0):
            some(f"length {t} with staging {st}", lambda c: c["target"] == t and c["staged"] == st and c["kind"] != "generic")
    # a chunk of 128 input frames adds ceil(128 q / p) outputs at most: how far each case lands from its edge
    for c in P:
        off = c["n_out"] - _target(c["target"], c["staged"])
        per_chunk = -(-128 * c["q"] // c["p"])
        assert (0 <= off < per_chunk) if c["target"] == "2tiles+1" else (-per_chunk < off <= 0), (c["name"], c["n_out"])
    some("a stream of exactly two tiles", lambda c: c["n_out"] == 2 * TILE)
    some("a stream of two tiles and one output", lambda c: c["n_out"] == 2 * TILE + 1)
    some("a stream that ends one output before a step boundary", lambda c: c["n_out"] % STEP == STEP - 1)
    for st in (2, 4):
        some(f"a stream that ends on a part boundary ({st} parts)",
             lambda c: c["staged"] == st and c["n_out"] % STEP == GEO["PART_MAX"][st] and c["kind"] != "generic")
    # staging by kind: unstaged (interior == 2: unchecked taps from global memory) and quarter-staged mono
    for kind in ("f32x1", "i16x1", "f32x2", "i16x2"):
        some(f"{kind} unstaged over several tiles", lambda c: c["kind"] == kind and c["staged"] == 0 and c["tiles"] >= 2)
        some(f"{kind} two-part staging", lambda c: c["kind"] == kind and c["staged"] == 2)
        some(f"{kind} quarter staging", lambda c: c["kind"] == kind and c["staged"] == 4)
        for pos in ("passthrough", "exact_q1", "exact_rational", "table_periodic", "table_rational", "table_q1"):
            some(f"{kind} {pos}", lambda c: c["kind"] == kind and c["pos"] == pos)
    # unstaged f32 stereo from just above 48 kHz, f32 mono and i16 stereo from about twice that
    assert min(c["rate"] for c in fast if c["kind"] == "f32x2" and c["staged"] == 0) <= 64000
    assert min(c["rate"] for c in fast if c["kind"] in ("f32x1", "i16x2") and c["staged"] == 0) <= 96200
    # the 48 kHz quad loops, mono and stereo (two-part and quarter staging)
    some("48 kHz f32 mono quad loop", lambda c: c["kind"] == "f32x1" and c["pos"] == "exact_48k")
    some("48 kHz f32 stereo quad loop", lambda c: c["kind"] == "f32x2" and c["pos"] == "exact_48k" and c["staged"] == 4)
    # periodic table at periods other than 44.1 kHz's 160, down to a period of 16 and up to KOFF_MAX
    qs = {c["q"] for c in P if c["pos"] == "table_periodic"}
    assert {16, 40, 80, 320, GEO["KOFF_MAX"]} <= qs, qs
    # the plain table path with periods far beyond KOFF_MAX
    some("table path with q > KOFF_MAX", lambda c: c["pos"] == "table_rational" and c["q"] > GEO["KOFF_MAX"] and c["kind"] != "generic")
    assert max(c["q"] for c in P if c["pos"] == "table_rational") >= 16000
    # up-sampling over more than one tile; q == 1 shortcut with p != 3; q == 1 with a table
    some("exact up-sampling over several tiles", lambda c: c["mode"] == RS_EXACT and c["p"] < c["q"] and c["tiles"] >= 2)
    assert {c["p"] for c in P if c["pos"] == "exact_q1"} >= {2, 4, 6, 12, 118}
    assert {c["p"] for c in P if c["pos"] == "table_q1"} >= {49, 93}
    # generic streams over several tiles, in both formats, with trailing partial frames
    for fmt in ("f32", "i16"):
        some(f"generic {fmt} over several tiles", lambda c: c["kind"] == "generic" and c["fmt"] == fmt and c["tiles"] >= 2)
    some("generic with a trailing partial frame", lambda c: c["kind"] == "generic" and c["drop"] > 0)
    some("stereo with a trailing partial frame", lambda c: c["ch"] == 2 and c["drop"] > 0)
    # the stage never reads past the last full 16 bytes: tails that are not a multiple of 16 bytes come through the checked path
    some("staged stream whose byte length is not a multiple of 16", lambda c: c["staged"] and c["nbytes"] % 16)
    # the 32-bit position math at the ratio guard (af_batch_create): within 1 % of 2^32
    span = TILE + GEO["YLEN"] + GEO["THREADS"]
    worst = max(c["p"] * span + c["q"] for c in P)
    assert 0.99 * 2 ** 32 <= worst < 2 ** 32, worst
    # the mixed batch: its first table rate has a period the periodic path serves; 44.1 kHz then takes the plain path
    first_table = next(c for c in P if c["mode"] == RS_TABLE)
    assert first_table["periodic"] and first_table["q"] != 160


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the fused kernel against the oracle
# ---------------------------------------------------------------------------------------------------------------------
_REF = {}


def _ref(orc, case):
    if case[0] not in _REF:
        x = _signal(case)
        _REF[case[0]] = (x, orc.pipeline_stream(x, case[3], case[2], orc.default_feat_config(80), orc.default_vad_config(),
                                                 400, 160, case[4]))
    return _REF[case[0]]


def _f32_rel_l2(orc, pcm, ref):
    """Relative L2 of a plain float32 log-mel of `pcm` (scipy's rfft in float32, float32 power and mel sums) against the
    f64 oracle's log-mel `ref` of the same PCM."""
    import scipy.fft
    cfg = orc.default_feat_config(ref.shape[1])
    fr = np.lib.stride_tricks.sliding_window_view(np.asarray(pcm, np.float32), 400)[::160][:len(ref)]
    X = scipy.fft.rfft(fr * orc.hann_window(400).astype(np.float32), 512, axis=1)
    P = X.real * X.real + X.imag * X.imag
    lm = np.log(np.maximum(P @ orc.mel_filterbank(cfg).astype(np.float32), np.float32(cfg.log_floor)))
    return float(np.sqrt(((lm.astype(np.float64) - ref) ** 2).sum() / (ref.astype(np.float64) ** 2).sum()))


def _assert_logmel(orc, got, ref, pcm, what):
    """assert_logmel_close's per-bin bound unchanged; its relative-L2 figure of 1e-5 is a property of broadband streams.
    Streams up-sampled from 4 or 8 kHz carry next to nothing above their input's Nyquist frequency, and there a float32
    transform is conditioning-limited on many bins: a plain float32 rfft of the very same (bit-exact) PCM lands at 5-6e-5.
    Beyond 1e-5 the kernel may be at most twice what that transform gives."""
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if ref.size == 0:
        return
    err = np.abs(got.astype(np.float64) - ref.astype(np.float64))
    tol = logmel_tolerance(ref)
    worst = np.unravel_index((err / tol).argmax(), err.shape)
    assert (err <= tol).all(), f"{what} logmel: err {err[worst]:.3e} > tol {tol[worst]:.3e} at {worst}"
    rel = float(np.sqrt((err ** 2).sum() / max((ref.astype(np.float64) ** 2).sum(), 1e-30)))
    if rel > LOGMEL_REL_L2:
        floor = _f32_rel_l2(orc, pcm, ref)
        assert rel <= 2.0 * floor, f"{what} logmel: rel L2 {rel:.3e}; a float32 rfft of the same PCM: {floor:.3e}"


def _check(orc, got, ref, what):
    """PCM, frame energies, VAD states and the final detector state bit-exact (_check_stream); log-mel by _assert_logmel."""
    _check_stream(dict(got, logmel=None), ref, what)
    if got.get("logmel") is not None and ref.get("logmel") is not None:
        _assert_logmel(orc, got["logmel"], ref["logmel"], ref["pcm"], what)


def _check_all(orc, results, what):
    """_check on every (case, got, ref); one failure report listing every stream that differs."""
    bad = []
    for case, got, ref in results:
        try:
            _check(orc, got, ref, f"{what} {case[0]}")
        except AssertionError as e:
            bad.append(str(e).splitlines()[0])
    assert not bad, f"{len(bad)} of {len(results)} streams differ:\n" + "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_each_case_alone(af, orc, case):
    """One stream per batch: a table rate gets the periodic path when its period allows, a two-part stream the kernel
    instance with a compile-time two parts per step."""
    x, ref = _ref(orc, case)
    got = af.Pipeline(af.pipeline_config(n_mels=80)).run_host([(x, case[2], case[3])])[0]
    assert len(got["pcm"]) == _geometry_of(case)[1]
    _check(orc, got, ref, case[0])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["sync", "tma"])
def test_mixed_batch(af, orc, variant):
    """Every case in one batch: the QUARTERS kernel instance for all, the periodic path for the first table rate only."""
    data = [_ref(orc, c) for c in CASES]
    try:
        af.set_kernel_variant(variant)
        got = af.Pipeline(af.pipeline_config(n_mels=80)).run_host([(x, c[2], c[3]) for c, (x, _) in zip(CASES, data)])
    finally:
        af.set_kernel_variant("auto")
    _check_all(orc, [(c, g, r) for c, (_, r), g in zip(CASES, data, got)], variant)


@pytest.mark.gpu
def test_mixed_batch_device_buffers_off_256(af, orc):
    """The mixed batch on device buffers, every stream 16 bytes past a 256-byte boundary (host mode rebases every
    stream to a 256-byte offset, so only device mode meets stage fills that start inside a 256-byte block)."""
    import torch
    dev = torch.device("cuda")
    data = [_ref(orc, c) for c in CASES]
    offs, pos = [], 0
    for x, _ in data:
        offs.append(pos + 16)
        pos += (x.nbytes + 16 + 255) // 256 * 256
    buf = torch.zeros(pos + 256, dtype=torch.uint8, device=dev)
    for (x, _), o in zip(data, offs):
        buf[o:o + x.nbytes].copy_(torch.from_numpy(np.ascontiguousarray(x).view(np.uint8)))
    base = buf.data_ptr()
    assert base % 256 == 0
    descs = [(base + o, x.size, c[2], c[3], af.AF_FMT_I16 if x.dtype == np.int16 else af.AF_FMT_F32)
             for c, (x, _), o in zip(CASES, data, offs)]
    b = af.Pipeline(af.pipeline_config(n_mels=80)).batch(descs, af.AF_MEM_DEVICE)
    S = len(CASES)
    pcm = torch.full((S, b.pcm_stride), float("nan"), device=dev)
    lm = torch.full((S, b.logmel_stride), float("nan"), device=dev)
    vad = torch.full((S, b.vad_stride), 255, device=dev, dtype=torch.uint8)
    en = torch.zeros((S, b.energy_stride), device=dev)
    fin = torch.zeros((S, 6), device=dev, dtype=torch.int32)
    o = b.outputs_struct(pcm.data_ptr(), b.pcm_stride, lm.data_ptr(), b.logmel_stride, vad.data_ptr(), b.vad_stride,
                         en.data_ptr(), b.energy_stride, fin.data_ptr())
    torch.cuda.synchronize()            # torch fills run on the legacy stream; the library uses its own non-blocking stream
    b.run_device(o)
    torch.cuda.synchronize()
    pcm, lm, vad, en, fin = pcm.cpu().numpy(), lm.cpu().numpy(), vad.cpu().numpy(), en.cpu().numpy(), fin.cpu().numpy()
    results = []
    for i, (c, (_, ref)) in enumerate(zip(CASES, data)):
        n_out, T = int(b.n_out[i]), int(b.n_feat[i])
        assert np.isnan(pcm[i, n_out:]).all(), c[0]                   # nothing past the stream's end is written
        got = {"pcm": pcm[i, :n_out], "logmel": lm[i, :T * 80].reshape(T, 80), "vad": vad[i, :T], "energy": en[i, :T],
               "vad_final": dict(state=int(fin[i, 1]), smoothed=float(fin[i, 0:1].view(np.float32)[0]), speech_frames=int(fin[i, 4]))}
        results.append((c, got, ref))
    _check_all(orc, results, "device")


def _check_specials(orc, case, got, x):
    ref = orc.resample_stream(orc.to_mono(orc.i16_to_f32(x) if x.dtype == np.int16 else x, case[3]), case[2])
    assert got.shape == ref.shape, case[0]
    nan = np.isnan(ref)
    assert (~nan).sum() > 0.5 * len(ref), case[0]
    assert np.array_equal(np.isnan(got), nan), f"{case[0]}: NaN positions differ"
    assert_bit_equal(got[~nan], ref[~nan], f"special values {case[0]}")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_special_values_alone(af, orc, case):
    """PCM only (as test_resampler_special_values): the shortcuts of every path stay bit-exact on the values that break
    them; NaN positions must match (payloads are implementation-defined)."""
    x = _specials(case)
    got = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False)).run_host([(x, case[2], case[3])])[0]["pcm"]
    _check_specials(orc, case, got, x)


@pytest.mark.gpu
def test_special_values_mixed_batch(af, orc):
    xs = [_specials(c) for c in CASES]
    got = af.Pipeline(af.pipeline_config(n_mels=0, vad_enable=False)).run_host([(x, c[2], c[3]) for c, x in zip(CASES, xs)])
    bad = []
    for c, x, g in zip(CASES, xs, got):
        try:
            _check_specials(orc, c, g["pcm"], x)
        except AssertionError as e:
            bad.append(str(e).splitlines()[0])
    assert not bad, f"{len(bad)} of {len(CASES)} streams differ:\n" + "\n".join(bad)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the same rates through the session kernel and the object resampler
# ---------------------------------------------------------------------------------------------------------------------
REALISTIC = [r for r in RATES if r <= 192000]


class _OneStream(Harness):
    """Harness (test_session_streams_gpu.py) whose whole-life log-mel check is _assert_logmel."""

    def close(self, k, vad_final=None, ended=False):
        L = self.life[k]
        pcm = np.concatenate(L.pcm) if L.pcm else np.zeros(0, np.float32)
        got = np.concatenate(L.lm) if L.lm else np.zeros((0, self.n_mels), np.float32)
        _assert_logmel(self.orc, got, self.orc.logmel(pcm, self.orc.default_feat_config(self.n_mels)), pcm, f"stream {k}")
        n_mels, self.n_mels = self.n_mels, 0                # the rest of Harness.close: VAD, detector state
        try:
            super().close(k, vad_final, ended)
        finally:
            self.n_mels = n_mels


@pytest.mark.gpu
@pytest.mark.parametrize("ch,fmt", KINDS, ids=[f"{f}x{c}" for c, f in KINDS])
@pytest.mark.parametrize("rate", REALISTIC)
def test_session_ragged_ticks(af, orc, rate, ch, fmt):
    """A one-stream Session: ragged ticks of up to 20 ms, one tick of a single frame mid-stream, end on the last tick;
    PCM bit-exact against the oracle's BatchResampler tick for tick, VAD and log-mel over the whole life."""
    max_frames = max(1, rate // 50)
    h = _OneStream(af, orc, 1, rate, ch, fmt, max_tick=max_frames * ch, seconds=1.5)
    rng = np.random.default_rng(rate + 7 * ch + (fmt == "i16"))
    n_ticks = 40
    for t in range(n_ticks):
        n = 1 if t == n_ticks // 2 else int(rng.integers(0, max_frames + 1))
        h.tick([n * ch], end=[t == n_ticks - 1])
    assert h.closed == 1                     # the end checked the stream's whole life: VAD, log-mel, detector state


@pytest.mark.gpu
@pytest.mark.parametrize("rate", REALISTIC + EXTREMES)
def test_batch_resampler_object(af, orc, rate):
    """BatchResampler.process / flush with random chunk sizes (as test_batch_resampler_matches_oracle)."""
    rng = np.random.default_rng(rate + 3)
    n = max(30000, 400 * (rate // OUT_RATE + 1) * 8)
    x = rng.standard_normal(n).astype(np.float32)
    x[rng.integers(0, n, 50)] = 0.0
    g, o = af.BatchResampler.new(rate, OUT_RATE), orc.BatchResampler(rate, OUT_RATE)
    pos, total = 0, 0
    while pos < len(x):
        k = int(rng.integers(1, 3000))
        a = g.process(x[pos:pos + k])
        assert_bit_equal(a, o.process(x[pos:pos + k]), f"process @ {pos}")
        pos, total = pos + k, total + len(a)
    assert_bit_equal(g.flush(), o.flush(), "flush")
    assert total > 200
