"""Stream records (af_session_export_streams, af_session_import_streams): a live stream exported from one session and
imported into a slot of another continues there exactly as if it had never moved.  Every moved caller is checked twice
on every tick: bitwise against a never-moved twin session of the same pipeline fed the same samples (PCM, states,
energies through the states, vad_final, log-mel, wire payloads and records, levels, first frames), and, through the twin's
harness, against the oracle objects whose life spans the move (bit-exact, log-mel within assert_logmel_close)."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

from test_parity_gpu import assert_bit_equal
from test_session_formats_gpu import FORMATS
from test_session_streams_gpu import Harness, _ragged_counts
from test_session_wire_gpu import _device_rows
from test_vad_configs_gpu import Configured, _configs


def _n_gpus():
    try:
        import audioflow
        n = C.c_int(0)
        audioflow.load_library().af_device_count(C.byref(n))
        return n.value
    except Exception:
        return 0


def _cuda_bytes(n, rb, device=0):
    import torch
    return torch.zeros((n, rb), dtype=torch.uint8, device=f"cuda:{device}")


class Fleet:
    """Callers c = 0..n-1 of the twin harness `h` (caller c in twin slot c, never moved) live in slots of `sessions`;
    where[c] = (session index, slot).  Every tick pushes the same samples to the twin and to each caller's current slot
    (idle slots push nothing) and compares every caller with its twin."""

    def __init__(self, af, h, sessions, where, levels=False, device_records=False):
        self.af, self.h, self.ses, self.where, self.levels = af, h, sessions, dict(where), levels
        self.device_records = device_records
        self.moves = 0
        if levels:
            for s in sessions:
                s.enable_levels()

    def _rows(self, si, xs, end):
        s = self.ses[si]
        f32 = s.fmt == self.af.AF_FMT_F32
        rows = [np.zeros(0, np.float32 if f32 else np.int16) for _ in range(s.S)]
        e = [False] * s.S
        for c, (sj, k) in self.where.items():
            if sj == si:
                x = xs[c]
                rows[k] = x.astype(np.float32) / np.float32(32768) if (f32 and x.dtype == np.int16) else x
                e[k] = bool(end[c]) if end is not None else False
        return rows, e

    def tick(self, counts, end=None):
        h = self.h
        xs = h.samples(counts)
        outs = [s.push_streams(*self._rows(si, xs, end)) for si, s in enumerate(self.ses)]
        wires = [s.wire() if s.wire_mem is not None else None for s in self.ses]
        lvs = [s.levels() if self.levels else None for s in self.ses]
        r = h.tick(counts, end, xs)
        wt = h.ses.wire() if h.wire is not None else None
        lt = h.ses.levels() if self.levels else None
        for c, (si, k) in self.where.items():
            if c not in h.check:
                continue
            o = outs[si]
            for key in ("pcm", "logmel", "vad"):
                assert_bit_equal(o[key][k], r[key][c], f"caller {c} {key}")
            for key in ("n_pcm", "n_feat", "n_vad"):
                assert int(o[key][k]) == int(r[key][c]), (c, key)
            assert o["vad_final"][k] == r["vad_final"][c], c
            if wt is not None and wires[si] is not None:
                w, a, b = wires[si], wires[si]["streams"][k], wt["streams"][c]
                assert int(w["first_frames"][k]) == int(wt["first_frames"][c]), c
                assert {q: v for q, v in a.items() if q not in ("pcm16", "base64")} == \
                       {q: v for q, v in b.items() if q not in ("pcm16", "base64")}, (c, a, b)
                if a["pcm16"] is None:
                    a = dict(a, pcm16=_device_rows(w["pcm16_ptr"], self.ses[si].S, w["pcm16_stride"], np.int16)[k, :a["n_samples"]],
                             base64=_device_rows(w["base64_ptr"], self.ses[si].S, w["base64_stride"], np.uint8)[k, :a["n_chars"]].tobytes())
                assert_bit_equal(a["pcm16"], b["pcm16"], f"caller {c} payload")
                assert a["base64"] == b["base64"], c
            if lt is not None:
                for key in ("level_db", "peak"):
                    assert lvs[si][key][k].view(np.uint32) == lt[key][c].view(np.uint32), (c, key)
                assert lvs[si]["is_speech"][k] == lt["is_speech"][c], c
        return r

    def free(self, si):
        used = {k for sj, k in self.where.values() if sj == si}
        return [k for k in range(self.ses[si].S) if k not in used]

    def move(self, callers, dst, slots, device=False):
        """Export `callers` from their sessions, import them into session `dst` at `slots`, reset the old slots."""
        by_src = {}
        for c, k in zip(callers, slots):
            by_src.setdefault(self.where[c][0], []).append((c, k))
        for si, pairs in by_src.items():
            src = self.ses[si]
            old = [self.where[c][1] for c, _ in pairs]
            rec = src.export_streams(old, out=_cuda_bytes(len(old), src.record_bytes()) if device else None)
            if device:
                import torch
                torch.cuda.synchronize()
            self.ses[dst].import_streams([k for _, k in pairs], rec)
            src.reset_streams(old)
            for c, k in pairs:
                self.where[c] = (dst, k)
        self.moves += len(callers)


def _hop(fleet, rng, frac=0.1):
    """A random `frac` of A's callers to random free slots of B, and as many of B's back to A."""
    for src, dst in ((0, 1), (1, 0)):
        mine = [c for c, (si, _) in fleet.where.items() if si == src]
        if not mine:
            continue
        pick = [int(c) for c in rng.choice(mine, max(1, int(len(mine) * frac)), replace=False)]
        slots = [int(k) for k in rng.choice(fleet.free(dst), len(pick), replace=False)]
        fleet.move(pick, dst, slots, device=bool(rng.integers(0, 2)) if fleet.device_records else False)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("framing", ["stft", "vad20"])
@pytest.mark.parametrize("wire_mem", ["host", "device"])
def test_callers_hop_between_sessions(af, orc, framing, wire_mem):
    """Sessions A and B admit the formats in different orders and with different bounds and sizes; ragged ticks; every
    few ticks 10 % of A's callers move to random free slots of B and as many back, through host and device records.
    Some callers have custom VAD configurations and B's pipeline has another default; gated wire on, levels on (STFT)."""
    mem = af.AF_MEM_HOST if wire_mem == "host" else af.AF_MEM_DEVICE
    rng = np.random.default_rng(31 + (framing == "stft") + 2 * (wire_mem == "host"))
    V = af.VadConfig
    if framing == "stft":
        n, fm = 20, FORMATS
        sf = [k % len(fm) for k in range(n)]
        cfgs = _configs(af)
        ccfg = [V() if k % 3 else cfgs[1 + k % (len(cfgs) - 1)] for k in range(n)]
        h = Configured(af, orc, fm, sf, ccfg, wire=(True, af.AF_MEM_HOST), levels=True, twins=False, seconds=8.0)
        pa = af.Pipeline(af.pipeline_config(n_mels=80))
        pb = af.Pipeline(af.pipeline_config(n_mels=80, vad=V(threshold_db=-35.0, min_speech_frames=1)))
        order_a = list(range(len(fm)))
        order_b = order_a[::-1]
        a = af.Session.formats(pa, [fm[i] for i in order_a], [0] * 24)
        b = af.Session.formats(pb, [(r, c, 2 * m) for r, c, m in (fm[i] for i in order_b)], [0] * 30)
        levels = True
    else:
        n = 12
        h = Harness(af, orc, n, 48000, max_tick=960, n_mels=0, vad_len=320, vad_hop=320, wire=(True, af.AF_MEM_HOST),
                    seconds=8.0)
        sf, fm, ccfg = [0] * n, [(48000, 1, 960)], None
        pa = af.Pipeline(af.pipeline_config(n_mels=0, vad_frame_len=320, vad_hop=320))
        pb = af.Pipeline(af.pipeline_config(n_mels=0, vad_frame_len=320, vad_hop=320, vad=V(threshold_db=-35.0)))
        a = af.Session.formats(pa, [(48000, 1, 960)], [0] * 16)
        b = af.Session.formats(pb, [(16000, 1, 320), (48000, 1, 1920)], [0] * 20)
        levels = False
    slots_a = [int(k) for k in rng.permutation(a.S)[:n]]
    for c in range(n):                                           # A's slots start in the callers' formats and configurations
        r_, ch_ = fm[sf[c]][:2]
        a.restart_streams([slots_a[c]], [next(j for j, f in enumerate(a.format_list) if f[:2] == (r_, ch_))])
    if ccfg is not None:
        custom = [c for c in range(n) if ccfg[c] != V()]
        a.set_vad_configs([slots_a[c] for c in custom], [ccfg[c] for c in custom])
    for s in (a, b):
        s.enable_wire(gate=True, mem=mem)
    fleet = Fleet(af, h, [a, b], {c: (0, slots_a[c]) for c in range(n)}, levels=levels, device_records=True)
    for t in range(36):
        counts = h.ragged(rng) if framing == "stft" else _ragged_counts(rng, n, 960, 1, t)
        r = fleet.tick(counts)
        if t % 3 == 2:
            _hop(fleet, rng)
    assert fleet.moves >= 20
    h.finish(r)


def _record_position(rec):
    """(last_index, chunks, n_out) of a record: StreamRecord's f64 bit pattern and counters after its first 32 bytes."""
    li = rec[32:40].copy().view(np.float64)[0]
    chunks, n_out = (int(v) for v in rec[40:56].copy().view(np.uint64))
    return li, chunks, n_out


@pytest.mark.gpu
@pytest.mark.parametrize("rate", [48000, 44100, 16000])
def test_positions_that_matter(af, orc, rate):
    """Residual 0 and 127 at the move; a caller moved on every tick (through segments: mid-segment, in Ending; the
    concatenated gated payload and records are checked over its whole life on finish); a pending restart after an end
    and after reset_streams; a stream that never pushed.  At 44.1 kHz the moved f64 position has drifted from the closed
    form, so a recomputed position would fail."""
    rng = np.random.default_rng(rate)
    n, mx = 6, rate // 50
    h = Harness(af, orc, n, rate, max_tick=mx, wire=(True, af.AF_MEM_HOST), levels=True, seconds=10.0)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a, b = (af.Session(pipe, 8, rate, 1, af.AF_FMT_F32, max_tick_samples=mx) for _ in range(2))
    for s in (a, b):
        s.enable_wire(gate=True)
    fleet = Fleet(af, h, [a, b], {c: (0, c) for c in range(n)}, levels=True)
    drifted = 0
    pushed = [0] * n
    for t in range(60):
        counts = [int(v) for v in rng.integers(1, mx + 1, n)]
        if rate != 16000:
            # caller 0 lands on residual 0 at tick 20 and caller 1 on residual 127 (input frames since the start)
            for c, res in ((0, 0), (1, 127)):
                if t == 19:
                    counts[c] = (res - pushed[c]) % 128 + 128 * int(rng.integers(0, (mx - 127) // 128 + 1))
        if t < 8:
            counts[5] = 0                                        # caller 5 never pushed before its move at tick 7
        end = [t == 14 and c == 3 for c in range(n)]
        for c in range(n):
            pushed[c] += counts[c]
        fleet.tick(counts, end)
        if t == 19 and rate != 16000:
            assert pushed[0] % 128 == 0 and pushed[1] % 128 == 127
        if t == 21:
            h.reset([4])
            fleet.ses[fleet.where[4][0]].reset_streams([fleet.where[4][1]])
        moving = [2] + [c for c, tt in ((0, 19), (1, 19), (3, 14), (4, 21), (5, 7)) if tt == t]
        for c in moving:
            si, k = fleet.where[c]
            if c == 2 and rate == 44100:
                li, chunks, n_out = _record_position(fleet.ses[si].export_streams([k])[0])
                exact = -4.0 + float(Fraction(n_out * 441, 160) - 128 * chunks)
                drifted += li != exact
            dst = 1 - si
            fleet.move([c], dst, [int(rng.choice(fleet.free(dst)))])
    if rate == 44100:
        assert drifted > 0
    h.finish(fleet.tick([0] * n))


@pytest.mark.gpu
def test_checkpoint_replay(af, orc):
    """Export every stream, push k ragged ticks, import the records back into the same slots and push the same k ticks:
    bit-identical outputs, the wire and levels included."""
    rng = np.random.default_rng(5)
    S = 6
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    s = af.Session.formats(pipe, FORMATS[:4], [k % 4 for k in range(S)])
    s.enable_wire(gate=True)
    s.enable_levels()
    src = [np.random.default_rng(k).standard_normal(48000 * 4 * 2).astype(np.float32) * 0.2 for k in range(S)]

    def ragged():
        return [int(rng.integers(0, FORMATS[k % 4][2] // FORMATS[k % 4][1] + 1)) * FORMATS[k % 4][1] for k in range(S)]

    pos = [0] * S
    for t in range(10):
        c = ragged()
        s.push_streams([src[k][pos[k]:pos[k] + c[k]] for k in range(S)])
        pos = [p + n for p, n in zip(pos, c)]
    rec = s.export_streams(range(S))
    assert (s.export_streams(range(S)) == rec).all()          # a snapshot does not change the session
    plan = [ragged() for _ in range(8)]
    passes = []
    for _ in range(2):
        out, p = [], list(pos)
        for c in plan:
            r = s.push_streams([src[k][p[k]:p[k] + c[k]] for k in range(S)], [t == 5 for t in range(S)])
            out.append((r, s.wire(), s.levels()))
            p = [a + n for a, n in zip(p, c)]
        passes.append(out)
        s.import_streams(range(S), rec)
        with pytest.raises(ValueError):
            s.wire()                                            # the last push no longer describes the slots
        with pytest.raises(ValueError):
            s.levels()
    for (r1, w1, l1), (r2, w2, l2) in zip(*passes):
        for key in ("pcm", "logmel", "vad"):
            for k in range(S):
                assert_bit_equal(r1[key][k], r2[key][k], key)
        assert r1["vad_final"] == r2["vad_final"]
        assert list(w1["first_frames"]) == list(w2["first_frames"])
        for a, b in zip(w1["streams"], w2["streams"]):
            assert {q: v for q, v in a.items() if q != "pcm16"} == {q: v for q, v in b.items() if q != "pcm16"}
            assert_bit_equal(a["pcm16"], b["pcm16"])
        for key in ("level_db", "peak"):
            assert (l1[key].view(np.uint32) == l2[key].view(np.uint32)).all()


@pytest.mark.gpu
def test_lockstep_session_into_a_fresh_one(af):
    """Every stream of a lockstep session imported into a fresh session of the same shape: its next push is the lockstep
    tick (4 launches) with outputs bitwise equal to the source's."""
    from audioflow import synth
    S, tick = 4, 960
    xs = np.stack([synth.stream(70 + i, 1.0, 48000, 1)[:tick * 20] for i in range(S)])
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    for t in range(7):
        a.push(xs[:, t * tick:(t + 1) * tick])
    b = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=tick)
    b.import_streams(range(S), a.export_streams(range(S)))
    for t in range(7, 12):
        x = xs[:, t * tick:(t + 1) * tick]
        ra = a.push(x)
        l0 = af.kernel_launch_count()
        rb = b.push(x)
        assert af.kernel_launch_count() - l0 == 4                # ingest+resample, fused (2), VAD scan
        assert "n_pcm" not in rb
        for key in ("pcm", "logmel", "vad"):
            assert_bit_equal(ra[key], rb[key], key)
        assert ra["vad_final"] == rb["vad_final"]


@pytest.mark.gpu
@pytest.mark.parametrize("src_fmt", ["f32", "i16"])
def test_wire_off_to_on_and_sample_types(af, orc, src_fmt):
    """Source wire off, destination wire on: the destination behaves as though enable_wire had been called at the import
    (the twin enables its wire then).  With src_fmt i16, an i16 session exports to an f32 one, whose caller pushes s / 32768."""
    rng = np.random.default_rng(8)
    n = 4
    h = Harness(af, orc, n, 48000, fmt=src_fmt, max_tick=960, seconds=6.0)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, 4, 48000, 1, af.AF_FMT_I16 if src_fmt == "i16" else af.AF_FMT_F32, max_tick_samples=960)
    b = af.Session(pipe, 6, 48000, 1, af.AF_FMT_F32, max_tick_samples=960)
    b.enable_wire(gate=True)
    fleet = Fleet(af, h, [a, b], {c: (0, c) for c in range(n)})
    for t in range(30):
        fleet.tick(_ragged_counts(rng, n, 960, 1, t))
        if t == 11:
            fleet.move(list(range(n)), 1, [5, 0, 3, 1])
            h.ses.enable_wire(gate=True)                         # the twin: enable_wire at the same point
            h.wire = (True, af.AF_MEM_HOST)
    h.wire = None                                                # (the harness's oracle check of the wire needs a whole life)
    h.finish(fleet.tick([0] * n))


@pytest.mark.gpu
def test_errors_leave_both_sessions_untouched(af, orc):
    """Every refused import and export is AF_ERR_INVALID and changes nothing: both sessions continue bit-exact."""
    rng = np.random.default_rng(12)
    n = 3
    h = Harness(af, orc, n, 48000, max_tick=960, wire=(True, af.AF_MEM_HOST), seconds=6.0)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session.formats(pipe, [(48000, 1, 960), (16000, 1, 320)], [0] * 4)
    b = af.Session.formats(pipe, [(16000, 1, 320), (48000, 1, 960)], [1] * 4)
    for s in (a, b):
        s.enable_wire(gate=True)
    fleet = Fleet(af, h, [a, b], {0: (0, 0), 1: (0, 1), 2: (1, 2)})
    L = af.load_library()
    u32p = C.POINTER(C.c_uint32)
    other = {  # sessions whose framing or formats do not match
        "framing": af.Session(af.Pipeline(af.pipeline_config(n_mels=0, vad_frame_len=320, vad_hop=320)), 2, 48000, 1),
        "no_vad": af.Session(af.Pipeline(af.pipeline_config(n_mels=80, vad_enable=False)), 2, 48000, 1),
        "format": af.Session(pipe, 2, 44100, 1),
    }

    def imp(ses, slots, rec, fmt=None, mem=af.AF_MEM_HOST):
        sl = np.array(slots, np.uint32)
        f = np.array(fmt, np.uint32) if fmt is not None else None
        return L.af_session_import_streams(ses._h, sl.ctypes.data_as(u32p), rec.ctypes.data if rec is not None else None,
                                           sl.size, f.ctypes.data_as(u32p) if f is not None else None, mem)

    for t in range(24):
        fleet.tick(_ragged_counts(rng, n, 960, 1, t))
        if t in (6, 15):
            rec = a.export_streams([0, 1])
            bad = []
            for off, val in ((0, 1), (4, 99), (8, 16)):          # magic, version, record size
                r = rec.copy()
                r[:, off:off + 4] = np.frombuffer(np.uint32(val).tobytes(), np.uint8)
                bad.append(r)
            for r in bad:
                assert imp(b, [0, 3], r) == af.AF_ERR_INVALID
            assert imp(b, [0, 4], rec) == af.AF_ERR_INVALID      # slot out of range
            assert imp(b, [3, 3], rec) == af.AF_ERR_INVALID      # slot listed twice
            assert imp(b, [0, 3], rec, [0, 1]) == af.AF_ERR_INVALID   # format 0 of b is 16 kHz
            assert imp(b, [0, 3], rec, [1, 2]) == af.AF_ERR_INVALID   # format index out of range
            assert imp(b, [0, 3], None) == af.AF_ERR_INVALID     # null records
            assert imp(b, [0, 3], rec, mem=7) == af.AF_ERR_INVALID
            for s in other.values():                             # framing 320/320, VAD off, 48 kHz not admitted
                r = np.zeros((2, s.record_bytes()), np.uint8)
                w = min(r.shape[1], rec.shape[1])
                r[:, :w] = rec[:, :w]
                r[:, 8:12] = np.frombuffer(np.uint32(s.record_bytes()).tobytes(), np.uint8)   # the size would pass
                assert imp(s, [0, 1], r) == af.AF_ERR_INVALID
            sl = np.array([0, 9], np.uint32)
            out = np.zeros((2, a.record_bytes()), np.uint8)
            assert L.af_session_export_streams(a._h, sl.ctypes.data_as(u32p), 2, out.ctypes.data, af.AF_MEM_HOST) == af.AF_ERR_INVALID
            assert L.af_session_export_streams(a._h, None, 2, out.ctypes.data, af.AF_MEM_HOST) == af.AF_ERR_INVALID
            assert L.af_session_export_streams(a._h, sl.ctypes.data_as(u32p), 1, out.ctypes.data, 7) == af.AF_ERR_INVALID
            assert not out.any()
            b.wire()                                             # no refused call spoiled the last push's outputs
        if t in (8, 17):
            c = [c for c, (si, _) in fleet.where.items() if si == 0][0]
            fleet.move([c], 1, [fleet.free(1)[0]])
    h.finish(fleet.tick([0] * n))


@pytest.mark.gpu
def test_scale_whole_session_move(af, orc):
    """1024 streams moved into a 2048-slot session at once (host records), then device records back into a third
    session; a seeded sample of 32 callers is checked against the twin and the oracle over 50 more ticks."""
    S = 1024
    rng = np.random.default_rng(2048)
    check = sorted(int(k) for k in rng.choice(S, 32, replace=False))
    h = Harness(af, orc, S, 48000, max_tick=1440, check=check, seconds=4.0)
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    a = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=1440)
    big = af.Session(pipe, 2 * S, 48000, 1, af.AF_FMT_F32, max_tick_samples=1440)
    fleet = Fleet(af, h, [a, big], {c: (0, c) for c in range(S)})
    for t in range(10):
        fleet.tick([int(v) for v in rng.integers(480, 1441, S)])
    # the whole session, checked and unchecked callers, into the larger one at shuffled slots
    slots = [int(k) for k in rng.permutation(2 * S)[:S]]
    rec = a.export_streams(range(S))
    big.import_streams(slots, rec)
    a.reset_streams(range(S))
    fleet.where = {c: (1, slots[c]) for c in range(S)}
    for t in range(25):
        r = fleet.tick([int(v) for v in rng.integers(480, 1441, S)])
    third = af.Session(pipe, S, 48000, 1, af.AF_FMT_F32, max_tick_samples=1440)
    fleet.ses.append(third)
    dev = big.export_streams(slots, out=_cuda_bytes(S, big.record_bytes()))
    import torch
    torch.cuda.synchronize()
    third.import_streams(range(S), dev)
    fleet.where = {c: (2, c) for c in range(S)}
    for t in range(25):
        r = fleet.tick([int(v) for v in rng.integers(480, 1441, S)])
    h.finish(r)


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs 2 GPUs")
def test_two_gpus(af, orc):
    """Export on GPU 0 (device records), copy to GPU 1, import there, continue bit-exact; and back through host records."""
    import torch
    rng = np.random.default_rng(2)
    n = 4
    af.init(0)
    h = Harness(af, orc, n, 44100, max_tick=882, wire=(True, af.AF_MEM_HOST), seconds=6.0)
    a = af.Session(h.pipe, 4, 44100, 1, af.AF_FMT_F32, max_tick_samples=882)
    af.init(1)
    b = af.Session(h.pipe, 6, 44100, 1, af.AF_FMT_F32, max_tick_samples=882)
    af.init(0)
    for s in (a, b):
        s.enable_wire(gate=True)
    fleet = Fleet(af, h, [a, b], {c: (0, c) for c in range(n)})
    for t in range(30):
        fleet.tick(_ragged_counts(rng, n, 882, 1, t))
        if t == 9:
            rec = a.export_streams(range(n), out=_cuda_bytes(n, a.record_bytes(), 0))
            torch.cuda.synchronize(0)
            rec1 = rec.to("cuda:1")
            torch.cuda.synchronize(1)
            b.import_streams([5, 1, 4, 0], rec1)
            a.reset_streams(range(n))
            fleet.where = {c: (1, k) for c, k in zip(range(n), [5, 1, 4, 0])}
        if t == 19:
            fleet.move(list(range(n)), 0, [3, 2, 1, 0])
    h.finish(fleet.tick([0] * n))


@pytest.mark.gpu
def test_resources(af):
    """Sessions that exported and imported free everything when destroyed; a second export of the same size allocates
    nothing."""
    import gc
    pipe = af.Pipeline(af.pipeline_config(n_mels=80))
    af.Session(pipe, 1, 48000, 1)                                # (the pipeline keeps its mel table on the device)
    gc.collect()
    base = af.live_allocations()
    a, b = (af.Session(pipe, 8, 48000, 1, af.AF_FMT_F32, max_tick_samples=960) for _ in range(2))
    a.push(np.zeros((8, 960), np.float32))
    rec = a.export_streams(range(8))
    mid = af.live_allocations()
    rec2 = a.export_streams(range(8))
    assert af.live_allocations() == mid and (rec == rec2).all()
    b.import_streams(range(8), rec)
    b.set_vad_configs([0], [af.VadConfig(threshold_db=-30.0)])
    b.import_streams([0], a.export_streams([1]))
    b.push(np.zeros((8, 960), np.float32))
    del a, b, rec, rec2
    gc.collect()
    assert af.live_allocations() == base


def test_python_argument_checks():
    """No GPU: export_streams / import_streams check their arguments before the library is called."""
    import audioflow as af

    class _Stub(af.Session):
        def __init__(self):
            self.S, self._h = 3, None
            self.format_list, self.stream_format = [(48000, 1, 960)], np.zeros(3, np.uint32)

        def record_bytes(self):
            return 64

    s = _Stub()
    with pytest.raises(ValueError):
        s.export_streams([0, 3])                                 # out of range
    with pytest.raises(ValueError):
        s.export_streams([-1])
    with pytest.raises(ValueError):
        s.import_streams([0, 0], np.zeros((2, 64), np.uint8))    # a slot listed twice
    with pytest.raises(ValueError):
        s.import_streams([0, 3], np.zeros((2, 64), np.uint8))
    with pytest.raises(ValueError):
        s.import_streams([0, 1], np.zeros((2, 63), np.uint8))    # truncated records
    with pytest.raises(ValueError):
        s.import_streams([0, 1], np.zeros((2, 64), np.int16))
    with pytest.raises(ValueError):
        s.import_streams([0], np.zeros((1, 64), np.uint8), format_ids=[1])   # format out of range
    with pytest.raises(ValueError):
        s.import_streams([0, 1], np.zeros((2, 64), np.uint8), format_ids=[0])
