"""CPU tests of the product's host side: the C-ABI library loads, exports every symbol the header
declares, fails loudly without a GPU, and its planning logic (output lengths, fractional-offset
plan, VAD threshold in the energy domain) agrees with the oracle.  No compute calls."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "audioflow_gpu.h")


def _declared_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"AF_API\s+[\w\s\*]+?\b(af_\w+)\s*\(", src)))


def test_library_loads_and_exports_header_symbols():
    import audioflow
    L = audioflow.load_library()
    syms = _declared_symbols()
    assert len(syms) >= 45
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing
    assert b"sm_100a" in L.af_version()


def test_no_gpu_fails_loudly():
    import audioflow
    L = audioflow.load_library()
    n = C.c_int(0)
    L.af_device_count(C.byref(n))
    if n.value > 0:
        pytest.skip("GPU present")
    with pytest.raises(audioflow.NoDevice) as e:
        audioflow.init()
    assert "no CPU fallback" in str(e.value)
    with pytest.raises(audioflow.NoDevice):
        audioflow.VoiceActivityDetector()
    with pytest.raises(audioflow.NoDevice):
        audioflow.AudioFrame.new([0.5, 0.25], 16000, 2).to_mono()
    with pytest.raises(audioflow.NoDevice):
        audioflow.AudioResampler(48000, 16000)


@pytest.mark.parametrize("rate", [48000, 44100, 32000, 22050, 8000, 16000, 96000, 11025])
def test_output_len_matches_oracle(orc, rate):
    import audioflow
    rng = np.random.default_rng(rate)
    lens = [0, 1, 127, 128, 129, 255, 256, 1000, 44100, 48000, 123457] + [int(v) for v in rng.integers(1, 300000, 6)]
    for n in lens:
        exp = len(orc.resample_stream(np.zeros(n, np.float32), rate))
        assert audioflow.resample_output_len(rate, 16000, n) == exp, (rate, n)


def test_output_len_tie_chunks_441(orc):
    """chunks = 193 mod 441 make (128 C - 8) * 160 / 441 an integer: the count hinges on f64 rounding."""
    import audioflow
    for chunks in (193, 193 + 441, 193 + 2 * 441):
        n = chunks * 128
        exp = len(orc.resample_stream(np.zeros(n, np.float32), 44100))
        assert audioflow.resample_output_len(44100, 16000, n) == exp


# 49 kHz: q = 16, a power of two, but the f64 step is not exactly 49 / 16; 784 kHz and 1.488 MHz: integer ratios (q = 1)
# whose f64 step is not exactly p either, so their fractions are not zero (at 1.488 MHz the recurrence sits just below
# every integer position)
@pytest.mark.parametrize("rate,mode", [(48000, 1), (44100, 2), (32000, 1), (22050, 2), (8000, 1), (24000, 1), (11025, 2),
                                       (49000, 2), (784000, 2), (1488000, 2)])
def test_resample_plan_fracs_match_oracle(orc, rate, mode):
    import audioflow
    L = audioflow.load_library()
    chunks = 400
    x = np.zeros(chunks * 128, np.float32)
    y, frac = orc.resample_stream(x, rate, return_frac=True)
    buf = np.empty(len(frac) + 16, np.float32)
    m = C.c_int(-1)
    n = L.af_debug_resample_plan(rate, 16000, chunks, buf.ctypes.data_as(C.POINTER(C.c_float)), len(buf), C.byref(m))
    assert n == len(frac)
    assert m.value == mode            # 1 = exact recurrence (dyadic step), 2 = table
    assert np.array_equal(buf[:n], frac)
    # exact positions: k = floor(P), rem/q; the oracle frac must be rem/q (exact) or within 1e-9 of it
    g = np.gcd(rate, 16000)
    p, q = rate // g, 16000 // g
    nn = np.arange(n, dtype=np.int64)
    num = (nn + 1) * p - 4 * q
    rem = np.mod(num, q)
    d = rem / q - frac.astype(np.float64)
    d = d - np.round(d)               # frac ~ 1 when the recurrence sits just below an integer
    assert np.max(np.abs(d)) < 1e-6
    if mode == 1:
        assert np.array_equal((rem / q).astype(np.float32), frac)


@pytest.mark.parametrize("thr", [-50.0, -40.0, -30.0, -60.5, -100.0, 0.0, 10.0, -50.000004])
def test_vad_threshold_in_energy_domain(orc, thr):
    import audioflow
    L = audioflow.load_library()
    e_min = np.float32(L.af_debug_vad_energy_threshold(thr))
    assert e_min > 0
    bits = int(e_min.view(np.uint32))
    # exhaustive neighbourhood: is_speech(e) == (e >= e_min) for 20000 floats either side
    for b in list(range(bits - 2000, bits + 2000)) + [bits - 10 ** 6, bits + 10 ** 6, 1, 0x7f7fffff]:
        e = np.uint32(b).view(np.float32)
        assert (orc.energy_to_dbfs(float(e)) > np.float32(thr)) == bool(e >= e_min), (b, e)
    assert not (orc.energy_to_dbfs(0.0) > thr)


def test_vad_threshold_edge_cases():
    import audioflow
    L = audioflow.load_library()
    assert np.isnan(L.af_debug_vad_energy_threshold(float("nan")))
    assert np.isnan(L.af_debug_vad_energy_threshold(float("inf")))
    tiny = np.float32(L.af_debug_vad_energy_threshold(float("-inf")))
    assert tiny.view(np.uint32) == 1          # any positive energy is speech; 0 is not


# ---- RingBuffer (capture.rs:84-161): the reference's own tests, capture.rs:425-515 and :547-560 ----
def test_ring_buffer_reference_tests():
    import threading
    import audioflow as af
    b = af.RingBuffer(1024)
    assert b.capacity == 1024                                             # test_ring_buffer_new
    assert b.write([1.0, 2.0, 3.0]) == 3                                  # test_ring_buffer_write_read
    assert b.read(3).tolist() == [1.0, 2.0, 3.0]
    b = af.RingBuffer(1024)                                               # test_ring_buffer_partial_read
    b.write([1.0, 2.0, 3.0, 4.0, 5.0])
    assert b.read(2).tolist() == [1.0, 2.0]
    assert b.read(3).tolist() == [3.0, 4.0, 5.0]
    b = af.RingBuffer(10)                                                 # test_ring_buffer_wrap_around
    b.write([1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0])
    b.read(5)
    b.write([8.0, 9.0, 10.0])
    assert b.read(5).tolist() == [6.0, 7.0, 8.0, 9.0, 10.0]
    b = af.RingBuffer(10)                                                 # test_ring_buffer_overflow: one slot stays free
    assert b.write([1.0] * 20) == 9
    r = b.read(9)
    assert len(r) == 9 and r.tolist() == [1.0] * 9
    assert af.RingBuffer(1024).read(100) is None                          # test_ring_buffer_read_empty
    b = af.RingBuffer(1024)                                               # test_ring_buffer_available
    assert b.available() == 0
    b.write([1.0] * 100)
    assert b.available() == 100
    b.read(50)
    assert b.available() == 50
    b.clear()                                                             # test_ring_buffer_clear
    assert b.available() == 0
    b = af.RingBuffer(1024)                                               # test_ring_buffer_thread_safe
    t = threading.Thread(target=lambda: b.write([1.0, 2.0, 3.0]))
    t.start(); t.join()
    assert b.read(3).tolist() == [1.0, 2.0, 3.0]


def test_ring_buffer_edges():
    import audioflow as af
    b = af.RingBuffer(4)
    assert b.write([]) == 0 and b.read(0) is None                          # empty ring: None even for read(0)
    assert b.write([1.0, 2.0, 3.0, 4.0]) == 3                              # capacity - 1 usable
    assert b.write([9.0]) == 0                                             # full: dropped
    assert len(b.read(0)) == 0                                             # Some(vec![]) on a non-empty ring
    assert b.read(10).tolist() == [1.0, 2.0, 3.0]
    # many wraps keep the order
    b = af.RingBuffer(7)
    nxt, got = 0.0, []
    for _ in range(50):
        w = b.write([nxt + i for i in range(5)])
        nxt += w
        got += b.read(3).tolist()
    assert got == [float(i) for i in range(len(got))]
    with pytest.raises(Exception):
        af.RingBuffer(0)                                                  # the reference would divide by zero on first use


# ---- the other host mirrors stay in step with the header ----
def test_cpp_mirror_compiles_against_the_header():
    """host/audioflow.hpp (the C++ stand-in for the Rust types) and its KAT program must compile against
    include/audioflow_gpu.h; running it needs a GPU, compiling it does not."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if not gxx:
        pytest.skip("no g++")
    host = os.path.join(ROOT, "audio-flow-rs_b200", "host")
    r = subprocess.run([gxx, "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "include"),
                        os.path.join(host, "test_reference_kat.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_rust_shim_binds_only_declared_symbols():
    """Every `pub fn af_*` of the Rust extern block (rust/src/ffi.rs; source only here: no Rust toolchain in the image)
    must be a symbol the header declares and the library exports."""
    ffi = open(os.path.join(ROOT, "audio-flow-rs_b200", "rust", "src", "ffi.rs")).read()
    names = set(re.findall(r"pub fn (af_[a-z0-9_]+)\s*\(", ffi))
    assert len(names) >= 20
    declared = set(_declared_symbols())
    missing = sorted(names - declared)
    assert not missing, f"ffi.rs binds symbols the header does not declare: {missing}"
