"""Python host-side mirror of the reference's audio module API
(src-tauri/src/modules/audio/mod.rs:9-11) on top of the C ABI of libaudioflow_gpu.so.

Same names, argument meaning and error behaviour as the Rust types, so that the parity tests
read like the reference's own `#[cfg(test)]` modules.  This file contains NO arithmetic of the
hot path: every call goes to the CUDA library and raises if it cannot be loaded or finds no GPU.
(The production host binding is the Rust shim under ../rust; Rust is not available in the build
image, see INTEGRATION.md.)
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from enum import IntEnum

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# AF_GPU_LIB selects another build of the same library (e.g. the `make STATS=1` debugging build)
LIB_PATH = os.environ.get("AF_GPU_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "libaudioflow_gpu.so")

AF_OK, AF_ERR_INVALID, AF_ERR_RESAMPLING_FAILED, AF_ERR_CUDA, AF_ERR_NO_DEVICE, AF_ERR_CAPACITY = range(6)
AF_FMT_F32, AF_FMT_I16 = 0, 1
AF_MEM_DEVICE, AF_MEM_HOST = 0, 1


class AudioError(Exception):
    """src-tauri/src/error.rs:96-111; only ResamplingFailed arises on this path."""


class ResamplingFailed(AudioError):
    def __init__(self, msg: str):
        super().__init__("Resampling failed: " + msg)
        self.msg = msg


class NoDevice(RuntimeError):
    pass


class _VadConfigC(C.Structure):
    _fields_ = [("threshold_db", C.c_float), ("smoothing_factor", C.c_float),
                ("silence_timeout_frames", C.c_uint64), ("min_speech_frames", C.c_uint64)]


class PipelineConfigC(C.Structure):
    _fields_ = [("n_mels", C.c_uint32), ("f_min", C.c_float), ("f_max", C.c_float), ("log_floor", C.c_float),
                ("log10", C.c_uint32), ("vad_enable", C.c_uint32), ("vad", _VadConfigC),
                ("vad_frame_len", C.c_uint32), ("vad_hop", C.c_uint32), ("write_pcm", C.c_uint32), ("pcm16", C.c_uint32)]


class StreamDescC(C.Structure):
    _fields_ = [("data", C.c_void_p), ("n_samples", C.c_uint64), ("sample_rate", C.c_uint32),
                ("channels", C.c_uint16), ("format", C.c_uint16)]


class VadFinalC(C.Structure):
    _fields_ = [("smoothed_energy", C.c_float), ("state", C.c_int32), ("silence_frames", C.c_uint64),
                ("speech_frames", C.c_uint64)]


class GateOutputsC(C.Structure):
    _fields_ = [("pcm", C.c_void_p), ("pcm_stride", C.c_uint64), ("logmel", C.c_void_p), ("logmel_stride", C.c_uint64),
                ("seg_offset", C.c_void_p), ("n_frames", C.c_void_p)]


class OutputsC(C.Structure):
    _fields_ = [("pcm", C.c_void_p), ("pcm_stride", C.c_uint64), ("logmel", C.c_void_p), ("logmel_stride", C.c_uint64),
                ("vad", C.c_void_p), ("vad_stride", C.c_uint64), ("energy", C.c_void_p), ("energy_stride", C.c_uint64),
                ("vad_final", C.c_void_p)]


class StreamFormatC(C.Structure):
    _fields_ = [("sample_rate", C.c_uint32), ("channels", C.c_uint16), ("pad", C.c_uint16), ("max_tick_samples", C.c_uint32)]


class WireConfigC(C.Structure):
    _fields_ = [("gate", C.c_uint32), ("pcm16", C.c_uint32), ("base64", C.c_uint32), ("mem", C.c_int32)]


class WireTickC(C.Structure):
    _fields_ = [("n_samples", C.c_uint32), ("n_chars", C.c_uint32), ("continued", C.c_uint32), ("started", C.c_uint16),
                ("ended", C.c_uint16), ("in_speech", C.c_uint8), ("pad", C.c_uint8 * 3)]


AF_MAX_GPUS = 16


class ShardedOutputsC(C.Structure):
    _fields_ = [("shard", OutputsC * AF_MAX_GPUS)]


_lib = None


def load_library():
    """Loads libaudioflow_gpu.so; raises if the extension was not built (no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(LIB_PATH)
    sz, fp, vp, u8p = C.c_size_t, C.POINTER(C.c_float), C.c_void_p, C.POINTER(C.c_uint8)
    szp = C.POINTER(sz)
    sig = {
        "af_init": (C.c_int, [C.c_int]), "af_shutdown": (C.c_int, []),
        "af_last_error": (sz, [C.c_char_p, sz]), "af_device_count": (C.c_int, [C.POINTER(C.c_int)]),
        "af_version": (C.c_char_p, []), "af_kernel_launch_count": (C.c_uint64, []),
        "af_debug_pipe_stats": (C.c_int, [C.POINTER(C.c_uint64)]),
        "af_debug_live_allocations": (C.c_int, [C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "af_host_alloc": (C.c_int, [C.POINTER(vp), sz]), "af_host_free": (C.c_int, [vp]),
        "af_to_mono": (C.c_int, [fp, sz, C.c_uint16, fp, sz, szp]),
        "af_resampler_create": (C.c_int, [C.c_uint32, C.c_uint32, C.POINTER(vp)]),
        "af_resampler_destroy": (None, [vp]),
        "af_resampler_process": (C.c_int, [vp, fp, sz, fp, sz, szp]),
        "af_resampler_input_rate": (C.c_uint32, [vp]), "af_resampler_output_rate": (C.c_uint32, [vp]),
        "af_resampler_needs_resampling": (C.c_int, [vp]), "af_resampler_chunk_size": (sz, [vp]),
        "af_resample_max_output": (sz, [C.c_uint32, C.c_uint32, sz]),
        "af_resample_output_len": (C.c_int, [C.c_uint32, C.c_uint32, sz, szp]),
        "af_batch_resampler_create": (C.c_int, [C.c_uint32, C.c_uint32, C.POINTER(vp)]),
        "af_batch_resampler_destroy": (None, [vp]),
        "af_batch_resampler_process": (C.c_int, [vp, fp, sz, fp, sz, szp]),
        "af_batch_resampler_flush": (C.c_int, [vp, fp, sz, szp]),
        "af_vad_config_default": (None, [C.POINTER(_VadConfigC)]),
        "af_vad_create": (C.c_int, [C.POINTER(_VadConfigC), C.POINTER(vp)]),
        "af_vad_destroy": (None, [vp]),
        "af_vad_detect": (C.c_int, [vp, fp, sz, u8p]),
        "af_vad_detect_frames": (C.c_int, [vp, fp, sz, C.c_uint32, C.c_uint32, u8p, sz, szp]),
        "af_vad_reset": (C.c_int, [vp]), "af_vad_state": (C.c_int, [vp]), "af_vad_energy_db": (C.c_float, [vp]),
        "af_vad_is_speaking": (C.c_int, [vp]), "af_vad_speech_frame_count": (C.c_uint64, [vp]),
        "af_vad_smoothed_energy": (C.c_float, [vp]),
        "af_vad_frame_energy": (C.c_int, [fp, sz, fp]),
        "af_pcm16_encode": (C.c_int, [fp, sz, C.POINTER(C.c_int16)]),
        "af_pcm16_base64_len": (C.c_size_t, [sz]),
        "af_pcm16_base64": (C.c_int, [fp, sz, C.c_char_p, sz, C.POINTER(C.c_size_t)]),
        "af_pipeline_config_default": (None, [C.POINTER(PipelineConfigC)]),
        "af_pipeline_create": (C.c_int, [C.POINTER(PipelineConfigC), C.POINTER(vp)]),
        "af_pipeline_destroy": (None, [vp]),
        "af_batch_create": (C.c_int, [vp, C.POINTER(StreamDescC), sz, C.c_int, C.POINTER(vp)]),
        "af_batch_destroy": (None, [vp]), "af_batch_n_streams": (sz, [vp]),
        "af_batch_counts": (C.c_int, [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "af_batch_strides": (C.c_int, [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "af_batch_run": (C.c_int, [vp, C.POINTER(OutputsC), vp]),
        "af_batch_run_host": (C.c_int, [vp, C.POINTER(OutputsC)]),
        "af_pipeline_run": (C.c_int, [vp, C.POINTER(StreamDescC), sz, C.POINTER(OutputsC)]),
        "af_set_kernel_variant": (C.c_int, [C.c_char_p]),
        "af_vad_segments": (C.c_int, [vp, C.c_uint64, vp, sz, vp, C.c_uint32, vp, vp]),
        "af_vad_gate": (C.c_int, [vp, C.c_uint64, vp, C.c_uint64, C.c_uint32, vp, C.c_uint32, vp, C.c_uint32, vp, sz,
                                  C.POINTER(GateOutputsC), vp]),
        "af_current_device": (C.c_int, []), "af_set_stream": (C.c_int, [vp]), "af_init_multi": (C.c_int, [C.c_int]),
        "af_comm_unique_id": (C.c_int, [u8p]), "af_comm_init_rank": (C.c_int, [C.c_int, C.c_int, u8p]),
        "af_comm_size": (C.c_int, []), "af_comm_shutdown": (C.c_int, []),
        "af_shard_partition": (C.c_int, [C.POINTER(StreamDescC), sz, C.c_int, szp]),
        "af_sharded_batch_create": (C.c_int, [vp, C.POINTER(StreamDescC), sz, C.c_int, C.POINTER(vp)]),
        "af_sharded_batch_destroy": (None, [vp]),
        "af_sharded_batch_shard": (C.c_int, [vp, C.c_int, szp, szp, C.POINTER(C.c_int)]),
        "af_sharded_batch_local": (vp, [vp, C.c_int]),
        "af_sharded_batch_run": (C.c_int, [vp, C.POINTER(ShardedOutputsC), C.c_int, C.c_int]),
        "af_sharded_batch_wait": (C.c_int, [vp]), "af_sharded_batch_join": (C.c_int, [vp]),
        "af_sharded_batch_gathered": (C.c_int, [vp, C.c_int, C.POINTER(vp), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                                C.POINTER(C.c_uint32)]),
        "af_sharded_batch_gathered_host": (C.c_int, [vp, C.c_int, u8p, C.c_uint64]),
        "af_sharded_batch_gather_ms": (C.c_int, [vp, C.c_int, fp]),
        "af_sharded_batch_run_host": (C.c_int, [vp, C.POINTER(OutputsC)]),
        "af_debug_vad_energy_threshold": (C.c_float, [C.c_float]),
        "af_debug_resample_plan": (sz, [C.c_uint32, C.c_uint32, sz, fp, sz, C.POINTER(C.c_int)]),
        "af_session_create": (C.c_int, [vp, sz, C.c_uint32, C.c_uint16, C.c_uint16, C.c_uint32, C.POINTER(vp)]),
        "af_session_destroy": (None, [vp]),
        "af_session_push": (C.c_int, [vp, vp, C.c_uint64, C.c_uint32, C.c_int, C.POINTER(OutputsC),
                                      C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "af_session_reset": (C.c_int, [vp]),
        "af_session_enable_levels": (C.c_int, [vp, C.c_int]),
        "af_session_levels": (C.c_int, [vp, fp, fp, u8p]),
        "af_session_enable_wire": (C.c_int, [vp, C.POINTER(WireConfigC)]),
        "af_session_wire": (C.c_int, [vp, C.POINTER(vp), C.POINTER(C.c_uint64), C.POINTER(vp), C.POINTER(C.c_uint64),
                                      C.POINTER(WireTickC), C.POINTER(C.c_uint64)]),
        "af_ring_create": (C.c_int, [sz, C.POINTER(vp)]), "af_ring_destroy": (None, [vp]),
        "af_ring_capacity": (sz, [vp]), "af_ring_write": (sz, [vp, fp, sz]),
        "af_ring_read": (C.c_int, [vp, fp, sz, szp]), "af_ring_available": (sz, [vp]), "af_ring_clear": (None, [vp]),
        "af_session_push_rings": (C.c_int, [vp, C.POINTER(vp), C.c_uint32, C.POINTER(OutputsC),
                                            C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "af_session_push_streams": (C.c_int, [vp, vp, C.c_uint64, C.POINTER(C.c_uint32), u8p, C.c_int, C.POINTER(OutputsC),
                                              C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "af_session_reset_streams": (C.c_int, [vp, C.POINTER(C.c_uint32), sz]),
        "af_session_push_rings_available": (C.c_int, [vp, C.POINTER(vp), C.c_uint32, u8p, C.POINTER(OutputsC),
                                                      C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
        "af_session_wire_first_frames": (C.c_int, [vp, C.POINTER(C.c_uint64)]),
        "af_session_create_formats": (C.c_int, [vp, sz, C.POINTER(StreamFormatC), sz, C.POINTER(C.c_uint32), C.c_uint16,
                                                C.POINTER(vp)]),
        "af_session_restart_streams": (C.c_int, [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), sz]),
        "af_batch_set_vad_configs": (C.c_int, [vp, C.POINTER(_VadConfigC)]),
        "af_session_set_vad_configs": (C.c_int, [vp, C.POINTER(C.c_uint32), C.POINTER(_VadConfigC), sz]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


EXPORTED_SYMBOLS = None  # filled lazily by tests from include/audioflow_gpu.h


def last_error() -> str:
    buf = C.create_string_buffer(1024)
    load_library().af_last_error(buf, 1024)
    return buf.value.decode("utf-8", "replace")


def _check(rc: int):
    if rc == AF_OK:
        return
    msg = last_error()
    if rc == AF_ERR_NO_DEVICE:
        raise NoDevice(msg)
    if rc in (AF_ERR_RESAMPLING_FAILED, AF_ERR_CUDA):
        raise ResamplingFailed(msg)          # the shim maps CUDA failures to the same variant
    if rc == AF_ERR_CAPACITY:
        raise BufferError(msg)
    raise ValueError(msg)


def init(device: int = -1):
    _check(load_library().af_init(device))


def kernel_launch_count() -> int:
    return int(load_library().af_kernel_launch_count())


def live_allocations() -> tuple[int, int]:
    """(device, pinned): the allocations the library holds right now (af_debug_live_allocations)."""
    d, p = C.c_uint64(0), C.c_uint64(0)
    _check(load_library().af_debug_live_allocations(C.byref(d), C.byref(p)))
    return int(d.value), int(p.value)


def set_kernel_variant(name: str):
    _check(load_library().af_set_kernel_variant(name.encode()))


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _fp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_float))


# ---------------------------------------------------------------------------------------------
# capture.rs:11-42
# ---------------------------------------------------------------------------------------------
@dataclass
class AudioFrame:
    samples: np.ndarray
    sample_rate: int
    channels: int
    timestamp_ns: int = 0

    @classmethod
    def new(cls, samples, sample_rate: int, channels: int, timestamp_ns: int = 0) -> "AudioFrame":
        return cls(_f32(samples), sample_rate, channels, timestamp_ns)

    def to_mono(self) -> "AudioFrame":
        """AudioFrame::to_mono (capture.rs:30-42), computed on the GPU."""
        x = _f32(self.samples)
        if self.channels == 1:
            return AudioFrame(x.copy(), self.sample_rate, 1, self.timestamp_ns)
        frames = (len(x) + self.channels - 1) // self.channels
        out = np.empty(frames, np.float32)
        n = C.c_size_t(0)
        _check(load_library().af_to_mono(_fp(x), len(x), self.channels, _fp(out), frames, C.byref(n)))
        return AudioFrame(out[:n.value], self.sample_rate, 1, self.timestamp_ns)


# ---------------------------------------------------------------------------------------------
# resampler.rs
# ---------------------------------------------------------------------------------------------
class AudioResampler:
    def __init__(self, input_rate: int, output_rate: int):
        h = C.c_void_p()
        _check(load_library().af_resampler_create(input_rate, output_rate, C.byref(h)))
        self._h = h

    @classmethod
    def new(cls, input_rate: int, output_rate: int) -> "AudioResampler":
        return cls(input_rate, output_rate)

    @classmethod
    def create_48k_to_16k(cls) -> "AudioResampler":
        return cls(48000, 16000)

    @classmethod
    def default(cls) -> "AudioResampler":
        return cls(48000, 16000)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_resampler_destroy(self._h)
            self._h = None

    def process(self, input) -> np.ndarray:
        x = _f32(input)
        out = np.empty(max(len(x), 512), np.float32)
        n = C.c_size_t(0)
        _check(load_library().af_resampler_process(self._h, _fp(x), len(x), _fp(out), len(out), C.byref(n)))
        return out[:n.value].copy()

    def input_rate(self) -> int: return int(load_library().af_resampler_input_rate(self._h))
    def output_rate(self) -> int: return int(load_library().af_resampler_output_rate(self._h))
    def needs_resampling(self) -> bool: return bool(load_library().af_resampler_needs_resampling(self._h))


class BatchResampler:
    def __init__(self, input_rate: int, output_rate: int):
        h = C.c_void_p()
        _check(load_library().af_batch_resampler_create(input_rate, output_rate, C.byref(h)))
        self._h = h
        self._rates = (input_rate, output_rate)

    @classmethod
    def new(cls, input_rate: int, output_rate: int) -> "BatchResampler":
        return cls(input_rate, output_rate)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_batch_resampler_destroy(self._h)
            self._h = None

    def process(self, input) -> np.ndarray:
        x = _f32(input)
        cap = load_library().af_resample_max_output(self._rates[0], self._rates[1], len(x) + 128)
        out = np.empty(cap, np.float32)
        n = C.c_size_t(0)
        _check(load_library().af_batch_resampler_process(self._h, _fp(x), len(x), _fp(out), cap, C.byref(n)))
        return out[:n.value].copy()

    def flush(self) -> np.ndarray:
        out = np.empty(1024, np.float32)
        n = C.c_size_t(0)
        _check(load_library().af_batch_resampler_flush(self._h, _fp(out), len(out), C.byref(n)))
        return out[:n.value].copy()


def resample_output_len(input_rate: int, output_rate: int, n_in: int) -> int:
    n = C.c_size_t(0)
    _check(load_library().af_resample_output_len(input_rate, output_rate, n_in, C.byref(n)))
    return int(n.value)


# ---------------------------------------------------------------------------------------------
# vad.rs
# ---------------------------------------------------------------------------------------------
class VadLevel(IntEnum):
    Aggressive = 0   # #[default]
    Balanced = 1
    Relaxed = 2


class VadState(IntEnum):
    Silence = 0
    Speech = 1
    Ending = 2


@dataclass
class VadConfig:
    threshold_db: float = -50.0
    smoothing_factor: float = 0.3
    silence_timeout_frames: int = 15
    min_speech_frames: int = 3

    def _c(self) -> _VadConfigC:
        return _VadConfigC(self.threshold_db, self.smoothing_factor, self.silence_timeout_frames,
                           self.min_speech_frames)


def _vad_config_array(cfgs):
    """A C array of the VadConfigs `cfgs` (ValueError for anything else, or a frame count outside uint64)."""
    cfgs = list(cfgs)
    for i, c in enumerate(cfgs):
        if not isinstance(c, VadConfig):
            raise ValueError(f"config {i} is not a VadConfig")
        for name in ("silence_timeout_frames", "min_speech_frames"):
            v = getattr(c, name)
            if not isinstance(v, (int, np.integer)) or not 0 <= int(v) < 1 << 64:
                raise ValueError(f"config {i}: {name} must be an integer in [0, 2^64)")
    return (_VadConfigC * max(len(cfgs), 1))(*[c._c() for c in cfgs])


class VoiceActivityDetector:
    def __init__(self, config: VadConfig | None = None):
        self.config = config if config is not None else VadConfig()
        h = C.c_void_p()
        c = self.config._c()
        _check(load_library().af_vad_create(C.byref(c), C.byref(h)))
        self._h = h

    @classmethod
    def new(cls, config: VadConfig) -> "VoiceActivityDetector":
        return cls(config)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_vad_destroy(self._h)
            self._h = None

    def detect(self, frame) -> VadState:
        f = _f32(frame)
        s = C.c_uint8(0)
        _check(load_library().af_vad_detect(self._h, _fp(f), len(f), C.byref(s)))
        return VadState(s.value)

    def detect_frames(self, samples, frame_len: int, hop: int) -> np.ndarray:
        x = _f32(samples)
        T = 1 + (len(x) - frame_len) // hop if len(x) >= frame_len else 0
        st = np.zeros(max(T, 1), np.uint8)
        n = C.c_size_t(0)
        _check(load_library().af_vad_detect_frames(self._h, _fp(x), len(x), frame_len, hop,
                                                   st.ctypes.data_as(C.POINTER(C.c_uint8)), len(st), C.byref(n)))
        return st[:n.value]

    def calculate_energy(self, frame) -> float:
        f = _f32(frame)
        e = C.c_float(0)
        _check(load_library().af_vad_frame_energy(_fp(f), len(f), C.byref(e)))
        return float(e.value)

    def reset(self): _check(load_library().af_vad_reset(self._h))
    def state(self) -> VadState: return VadState(load_library().af_vad_state(self._h))
    def energy_db(self) -> float: return float(load_library().af_vad_energy_db(self._h))
    def is_speaking(self) -> bool: return bool(load_library().af_vad_is_speaking(self._h))
    def speech_frame_count(self) -> int: return int(load_library().af_vad_speech_frame_count(self._h))
    def smoothed_energy(self) -> float: return float(load_library().af_vad_smoothed_energy(self._h))


def pcm16_encode(samples) -> np.ndarray:
    x = _f32(samples)
    out = np.empty(len(x), np.int16)
    _check(load_library().af_pcm16_encode(_fp(x), len(x), out.ctypes.data_as(C.POINTER(C.c_int16))))
    return out


def pcm16_base64(samples) -> bytes:
    """The "audio_base_64" payload of WebSocketClient::send_audio (websocket.rs:244-254): base64 of the PCM16 LE bytes."""
    L = load_library()
    x = _f32(samples)
    cap = int(L.af_pcm16_base64_len(len(x)))
    buf = C.create_string_buffer(max(cap, 1))
    n = C.c_size_t(0)
    _check(L.af_pcm16_base64(_fp(x), len(x), buf, cap, C.byref(n)))
    return buf.raw[:n.value]


# ---------------------------------------------------------------------------------------------
# batched pipeline
# ---------------------------------------------------------------------------------------------
def pipeline_config(n_mels: int = 80, vad: VadConfig | None = None, vad_enable: bool = True, vad_frame_len: int = 0,
                    vad_hop: int = 0, write_pcm: bool = True, log10: bool = False, f_min: float = 0.0,
                    f_max: float = 8000.0, log_floor: float = 1e-10, pcm16: bool = False) -> PipelineConfigC:
    c = PipelineConfigC()
    load_library().af_pipeline_config_default(C.byref(c))
    c.n_mels = n_mels
    c.f_min, c.f_max, c.log_floor, c.log10 = f_min, f_max, log_floor, int(log10)
    c.vad_enable = int(vad_enable)
    if vad is not None:
        c.vad = vad._c()
    c.vad_frame_len, c.vad_hop = vad_frame_len, vad_hop
    c.write_pcm = int(write_pcm)
    c.pcm16 = int(pcm16)
    return c


class Pipeline:
    def __init__(self, cfg: PipelineConfigC | None = None):
        self.cfg = cfg if cfg is not None else pipeline_config()
        h = C.c_void_p()
        _check(load_library().af_pipeline_create(C.byref(self.cfg), C.byref(h)))
        self._h = h

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_pipeline_destroy(self._h)
            self._h = None

    def batch(self, descs, mem: int) -> "Batch":
        return Batch(self, descs, mem)

    def run_host(self, streams):
        """streams: list of (ndarray samples [f32 or i16, interleaved], sample_rate, channels).
        Returns a list of dicts(pcm, logmel, vad, energy, vad_final) -- the reference-facing call with HOST buffers."""
        arrays, descs = [], []
        for (x, rate, ch) in streams:
            if x.dtype == np.int16:
                a, fmt = np.ascontiguousarray(x), AF_FMT_I16
            else:
                a, fmt = _f32(x), AF_FMT_F32
            arrays.append(a)
            descs.append((a.ctypes.data, a.size, rate, ch, fmt))
        b = Batch(self, descs, AF_MEM_HOST)
        out = b.alloc_host_outputs()
        b.run_host(out)
        return b.split(out)


def _desc_array(descs):
    arr = (StreamDescC * max(len(descs), 1))()
    for i, (ptr, n_samples, rate, ch, fmt) in enumerate(descs):
        arr[i] = StreamDescC(ptr or None, n_samples, rate, ch, fmt)
    return arr


class Batch:
    def __init__(self, pipe: Pipeline, descs, mem: int, _handle=None, _n=None):
        self.pipe = pipe
        self._owned = _handle is None
        if _handle is None:
            self.n = len(descs)
            h = C.c_void_p()
            _check(load_library().af_batch_create(pipe._h, _desc_array(descs), self.n, mem, C.byref(h)))
        else:                       # a shard of a ShardedBatch: the sharded batch owns the handle
            self.n, h = _n, C.c_void_p(_handle)
        self._h = h
        self.mem = mem
        self.n_out = np.zeros(max(self.n, 1), np.uint32)
        self.n_feat = np.zeros(max(self.n, 1), np.uint32)
        self.n_vad = np.zeros(max(self.n, 1), np.uint32)
        u32p = C.POINTER(C.c_uint32)
        _check(load_library().af_batch_counts(h, self.n_out.ctypes.data_as(u32p), self.n_feat.ctypes.data_as(u32p),
                                              self.n_vad.ctypes.data_as(u32p)))
        ps, ls, vs = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        _check(load_library().af_batch_strides(h, C.byref(ps), C.byref(ls), C.byref(vs)))
        self.pcm_stride, self.logmel_stride, self.vad_stride = ps.value, ls.value, vs.value
        self.energy_stride = (max(int(self.n_vad.max()) if self.n else 0, 4) + 3) // 4 * 4

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None and getattr(self, "_owned", True):
            _lib.af_batch_destroy(self._h)
            self._h = None

    def alloc_host_outputs(self) -> dict:
        cfg = self.pipe.cfg
        n = max(self.n, 1)
        out = {"pcm": np.zeros((n, self.pcm_stride), np.int16 if cfg.pcm16 else np.float32) if cfg.write_pcm else None,
               "logmel": np.zeros((n, self.logmel_stride), np.float32) if cfg.n_mels else None,
               "vad": np.zeros((n, self.vad_stride), np.uint8) if cfg.vad_enable else None,
               "energy": np.zeros((n, self.energy_stride), np.float32) if cfg.vad_enable else None,
               "vad_final": (VadFinalC * n)() if cfg.vad_enable else None}
        return out

    @staticmethod
    def outputs_struct(pcm=0, pcm_stride=0, logmel=0, logmel_stride=0, vad=0, vad_stride=0, energy=0, energy_stride=0,
                       vad_final=0) -> OutputsC:
        return OutputsC(pcm or None, pcm_stride, logmel or None, logmel_stride, vad or None, vad_stride,
                        energy or None, energy_stride, vad_final or None)

    def _host_struct(self, out: dict) -> OutputsC:
        def ptr(a):
            return a.ctypes.data if a is not None else 0
        return self.outputs_struct(ptr(out["pcm"]), self.pcm_stride, ptr(out["logmel"]), self.logmel_stride,
                                   ptr(out["vad"]), self.vad_stride, ptr(out["energy"]), self.energy_stride,
                                   C.addressof(out["vad_final"]) if out["vad_final"] is not None else 0)

    def run_host(self, out: dict):
        o = self._host_struct(out)
        _check(load_library().af_batch_run_host(self._h, C.byref(o)))

    def run_device(self, o: OutputsC, cuda_stream: int = 0):
        _check(load_library().af_batch_run(self._h, C.byref(o), cuda_stream or None))

    def set_vad_configs(self, cfgs):
        """One VadConfig per stream (VoiceActivityDetector::new(config) per caller) from the next run; None: the
        pipeline's for every stream."""
        if not self.pipe.cfg.vad_enable:
            raise ValueError("the pipeline runs no VAD (vad_enable == 0)")
        if cfgs is None:
            _check(load_library().af_batch_set_vad_configs(self._h, None))
            return
        cfgs = list(cfgs)
        if len(cfgs) != self.n:
            raise ValueError(f"{len(cfgs)} configs for {self.n} streams")
        _check(load_library().af_batch_set_vad_configs(self._h, _vad_config_array(cfgs)))

    def split(self, out: dict) -> list:
        res = []
        M = self.pipe.cfg.n_mels
        for i in range(self.n):
            r = {"pcm": None, "logmel": None, "vad": None, "energy": None, "vad_final": None}
            if out["pcm"] is not None:
                r["pcm"] = out["pcm"][i, :self.n_out[i]].copy()
            if out["logmel"] is not None:
                T = int(self.n_feat[i])
                r["logmel"] = out["logmel"][i, :T * M].reshape(T, M).copy()
            if out["vad"] is not None:
                r["vad"] = out["vad"][i, :self.n_vad[i]].copy()
                r["energy"] = out["energy"][i, :self.n_vad[i]].copy()
                f = out["vad_final"][i]
                r["vad_final"] = dict(state=int(f.state), smoothed=float(f.smoothed_energy),
                                      speech_frames=int(f.speech_frames), silence_frames=int(f.silence_frames))
            res.append(r)
        return res


# ---------------------------------------------------------------------------------------------
# multi-GPU: stream sharding + NCCL result gather behind the C ABI (SURVEY.md 8(e))
# ---------------------------------------------------------------------------------------------
def init_multi(n_gpus: int = 0):
    """ONE process drives GPUs 0..n-1 (ncclCommInitAll inside the library)."""
    _check(load_library().af_init_multi(n_gpus))


def comm_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    _check(load_library().af_comm_unique_id(buf))
    return bytes(buf)


def comm_init_rank(n_ranks: int, rank: int, uid: bytes | None):
    buf = (C.c_uint8 * 128)(*uid) if uid is not None else None
    _check(load_library().af_comm_init_rank(n_ranks, rank, buf))


def comm_shutdown():
    _check(load_library().af_comm_shutdown())


def shard_partition(descs, n_shards: int):
    """Contiguous blocks of stream indices balanced by input bytes: list of (lo, hi)."""
    first = (C.c_size_t * (n_shards + 1))()
    _check(load_library().af_shard_partition(_desc_array(descs), len(descs), n_shards, first))
    return [(int(first[r]), int(first[r + 1])) for r in range(n_shards)]


class ShardedBatch:
    """n global streams over the ranks of the communicator; this process runs the shards of the ranks it owns."""

    def __init__(self, pipe: Pipeline, descs, mem: int):
        self.pipe, self.n, self.mem = pipe, len(descs), mem
        h = C.c_void_p()
        _check(load_library().af_sharded_batch_create(pipe._h, _desc_array(descs), self.n, mem, C.byref(h)))
        self._h = h
        self.n_ranks = max(int(load_library().af_comm_size()), 1)

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_sharded_batch_destroy(self._h)
            self._h = None

    def shard(self, rank: int):
        """(first, count, device) -- device is -1 when another process owns the rank."""
        a, b, d = C.c_size_t(0), C.c_size_t(0), C.c_int(-1)
        _check(load_library().af_sharded_batch_shard(self._h, rank, C.byref(a), C.byref(b), C.byref(d)))
        return int(a.value), int(b.value), int(d.value)

    def local(self, rank: int) -> Batch | None:
        h = load_library().af_sharded_batch_local(self._h, rank)
        if not h:
            return None
        return Batch(self.pipe, None, self.mem, _handle=h, _n=self.shard(rank)[1])

    def run(self, outs: ShardedOutputsC, gather: bool = True, wait: bool = True):
        _check(load_library().af_sharded_batch_run(self._h, C.byref(outs), int(gather), 0 if wait else 1))

    def wait(self):
        _check(load_library().af_sharded_batch_wait(self._h))

    def join(self):
        _check(load_library().af_sharded_batch_join(self._h))

    def gathered(self, rank: int):
        """(device pointer, row stride, rows per rank, n_vad_frames[n]) of the last gather on a local rank's GPU."""
        p, st, rows = C.c_void_p(), C.c_uint64(0), C.c_uint64(0)
        nv = np.zeros(max(self.n, 1), np.uint32)
        _check(load_library().af_sharded_batch_gathered(self._h, rank, C.byref(p), C.byref(st), C.byref(rows),
                                                        nv.ctypes.data_as(C.POINTER(C.c_uint32))))
        return p.value, int(st.value), int(rows.value), nv[:self.n]

    def gathered_host(self, rank: int) -> np.ndarray:
        """[n_streams, stride] u8 states of ALL streams, global order, copied from the rank's GPU."""
        _, _, _, nv = self.gathered(rank)
        stride = (max(int(nv.max()) if self.n else 0, 16) + 15) // 16 * 16
        out = np.zeros((max(self.n, 1), stride), np.uint8)
        _check(load_library().af_sharded_batch_gathered_host(self._h, rank, out.ctypes.data_as(C.POINTER(C.c_uint8)), stride))
        return out[:self.n]

    def gather_ms(self, rank: int) -> float:
        ms = C.c_float(0)
        _check(load_library().af_sharded_batch_gather_ms(self._h, rank, C.byref(ms)))
        return float(ms.value)

    def run_host(self, o: OutputsC):
        _check(load_library().af_sharded_batch_run_host(self._h, C.byref(o)))


# ---------------------------------------------------------------------------------------------
# streaming sessions (BASELINE config 5)
# ---------------------------------------------------------------------------------------------
def stream_rows(xs, n_streams: int, channels, dtype):
    """The rows of a ragged tick: xs[k] (1-D interleaved samples of stream k) at the start of row k of one [n_streams,
    stride] array -> (array, uint32 counts).  channels: one count for all streams, or one per stream.  ValueError before
    anything is pushed for a wrong stream count, a row that is not 1-D, or a partial frame."""
    if len(xs) != n_streams:
        raise ValueError(f"{len(xs)} arrays for {n_streams} streams")
    ch = np.broadcast_to(np.asarray(channels, np.int64), (n_streams,))
    xs = [np.ascontiguousarray(x, dtype=dtype) for x in xs]
    for k, x in enumerate(xs):
        if x.ndim != 1:
            raise ValueError(f"stream {k}: samples must be 1-D (interleaved), got shape {x.shape}")
        if x.size % ch[k]:
            raise ValueError(f"stream {k}: {x.size} samples are not a whole number of {ch[k]}-channel frames")
    counts = np.array([x.size for x in xs], np.uint32)
    buf = np.zeros((n_streams, max((int(counts.max()) + 3) // 4 * 4, 4)), dtype)
    for k, x in enumerate(xs):
        buf[k, :x.size] = x
    return buf, counts


def end_flags(end, n_streams: int):
    """None, or one flag per stream as uint8 (ValueError for any other length)."""
    if end is None:
        return None
    e = np.ascontiguousarray(end, dtype=bool).astype(np.uint8).reshape(-1)
    if e.size != n_streams:
        raise ValueError(f"{e.size} end flags for {n_streams} streams")
    return e


class Session:
    """n_streams lockstep streams with persistent device state (resampler position + residual input,
    STFT overlap, VAD).  push() takes host arrays [n_streams, n_samples] and returns per-tick outputs.
    push_streams() / push_rings_available() / reset_streams() give every stream its own timeline.
    Session.formats() builds a session whose streams each have their own capture format; restart_streams() moves a
    stream to another one."""

    def __init__(self, pipe: Pipeline, n_streams: int, sample_rate: int, channels: int = 1, fmt: int = AF_FMT_F32,
                 max_tick_samples: int = 4096):
        h = C.c_void_p()
        _check(load_library().af_session_create(pipe._h, n_streams, sample_rate, channels, fmt, max_tick_samples, C.byref(h)))
        self._setup(pipe, h, [(sample_rate, channels, max_tick_samples)], np.zeros(n_streams, np.uint32), fmt)

    @classmethod
    def formats(cls, pipe: Pipeline, formats, stream_format, fmt: int = AF_FMT_F32) -> "Session":
        """A session of len(stream_format) streams that admits `formats`, a list of (sample_rate, channels,
        max_tick_samples); stream k starts in formats[stream_format[k]].  fmt (f32 / i16 samples) is the same for all."""
        formats = [tuple(int(v) for v in f) for f in formats]
        sf = np.ascontiguousarray(stream_format, dtype=np.uint32).reshape(-1)
        if any(len(f) != 3 for f in formats):
            raise ValueError("a format is (sample_rate, channels, max_tick_samples)")
        arr = (StreamFormatC * max(len(formats), 1))(*[StreamFormatC(r, c, 0, m) for r, c, m in formats])
        h = C.c_void_p()
        _check(load_library().af_session_create_formats(pipe._h, sf.size, arr, len(formats),
                                                        sf.ctypes.data_as(C.POINTER(C.c_uint32)), fmt, C.byref(h)))
        self = cls.__new__(cls)
        self._setup(pipe, h, formats, sf.copy(), fmt)
        return self

    def _setup(self, pipe, h, formats, stream_format, fmt):
        self.pipe, self._h, self.S, self.fmt = pipe, h, stream_format.size, fmt
        self.format_list = formats                      # (sample_rate, channels, max_tick_samples) per format
        self.stream_format = stream_format              # each stream's current format (restart_streams changes it)
        # a single-format session keeps its rate and channel count as attributes
        self.rate, self.channels = formats[0][:2] if len(formats) == 1 else (None, None)
        L = load_library()
        self.max_pcm = max(L.af_resample_max_output(r, 16000, m // c + 128) + 8 for r, c, m in formats)
        self.max_T = self.max_pcm // 160 + 4
        self.wire_mem = None                            # where the wire rows live (enable_wire)

    def stream_channels(self) -> np.ndarray:
        """The channel count of every stream's current format."""
        return np.array([self.format_list[f][1] for f in self.stream_format], np.int64)

    def _check_frames(self, n: int):
        ch = self.stream_channels()
        bad = np.nonzero(n % ch)[0]
        if bad.size:
            k = int(bad[0])
            raise ValueError(f"stream {k}: {n} samples are not a whole number of {ch[k]}-channel frames")

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_session_destroy(self._h)
            self._h = None

    def reset(self):
        _check(load_library().af_session_reset(self._h))

    def _run(self, call):
        cfg = self.pipe.cfg
        M = max(cfg.n_mels, 1)
        pcm = np.zeros((self.S, (self.max_pcm + 3) // 4 * 4), np.float32)
        lm = np.zeros((self.S, (self.max_T * M + 3) // 4 * 4), np.float32)
        vad = np.zeros((self.S, (self.max_T + 15) // 16 * 16), np.uint8)
        fin = (VadFinalC * self.S)()
        o = OutputsC(pcm.ctypes.data if cfg.write_pcm else None, pcm.shape[1], lm.ctypes.data if cfg.n_mels else None,
                     lm.shape[1], vad.ctypes.data if cfg.vad_enable else None, vad.shape[1], None, 0,
                     C.addressof(fin) if cfg.vad_enable else None)
        u32p = C.POINTER(C.c_uint32)
        npcm, nf, nv = (np.zeros(self.S, np.uint32) for _ in range(3))
        _check(call(C.byref(o), npcm.ctypes.data_as(u32p), nf.ctypes.data_as(u32p), nv.ctypes.data_as(u32p)))
        final = [dict(state=int(f.state), smoothed=float(f.smoothed_energy), speech_frames=int(f.speech_frames)) for f in fin]
        return pcm, lm, vad, npcm, nf, nv, final, M

    def _tick(self, call) -> dict:
        """Lockstep form: [n_streams, n] arrays.  When the streams emitted different counts (their timelines have
        diverged through push_streams / reset_streams), the per-stream form of push_streams instead: r["pcm"][k] etc. are
        stream k's own outputs either way."""
        pcm, lm, vad, npcm, nf, nv, final, M = self._run(call)
        if (npcm != npcm[0]).any() or (nf != nf[0]).any() or (nv != nv[0]).any():
            return self._per_stream(pcm, lm, vad, npcm, nf, nv, final, M)
        T = int(max(nf[0], nv[0]))
        return {"pcm": pcm[:, :npcm[0]].copy(), "logmel": lm[:, :int(nf[0]) * M].reshape(self.S, int(nf[0]), M).copy(),
                "vad": vad[:, :int(nv[0])].copy(), "n_frames": T, "vad_final": final}

    def _tick_streams(self, call) -> dict:
        return self._per_stream(*self._run(call))

    def _per_stream(self, pcm, lm, vad, npcm, nf, nv, final, M) -> dict:
        """Per-stream lists: stream k's own pcm / logmel [n_feat[k], n_mels] / vad, the counts and vad_final."""
        return {"pcm": [pcm[k, :npcm[k]].copy() for k in range(self.S)],
                "logmel": [lm[k, :int(nf[k]) * M].reshape(int(nf[k]), M).copy() for k in range(self.S)],
                "vad": [vad[k, :nv[k]].copy() for k in range(self.S)],
                "n_pcm": npcm, "n_feat": nf, "n_vad": nv, "vad_final": final}

    def push(self, x: np.ndarray) -> dict:
        """Every stream pushes x[k]; on a session whose streams have diverged the result may take the per-stream form
        (see _tick)."""
        x = np.ascontiguousarray(x, dtype=np.int16 if self.fmt == AF_FMT_I16 else np.float32)
        assert x.ndim == 2 and x.shape[0] == self.S
        n = x.shape[1]
        self._check_frames(n)
        L = load_library()
        return self._tick(lambda o, a, b, c: L.af_session_push(self._h, x.ctypes.data, n, n, AF_MEM_HOST, o, a, b, c))

    def enable_levels(self, on: bool = True):
        _check(load_library().af_session_enable_levels(self._h, 1 if on else 0))

    def levels(self) -> dict:
        """AudioLevel / VolumeLevel payloads of the last tick: level_db (energy_db()), peak (max |y|), is_speech."""
        lv, pk, sp = np.zeros(self.S, np.float32), np.zeros(self.S, np.float32), np.zeros(self.S, np.uint8)
        _check(load_library().af_session_levels(self._h, lv.ctypes.data_as(C.POINTER(C.c_float)),
                                                pk.ctypes.data_as(C.POINTER(C.c_float)), sp.ctypes.data_as(C.POINTER(C.c_uint8))))
        return {"level_db": lv, "peak": pk, "is_speech": sp.astype(bool)}

    def push_rings(self, rings, n_samples: int) -> dict:
        """One tick fed by the capture rings (AudioCapturer::read_frame for every stream, capture.rs:310-319)."""
        assert len(rings) == self.S
        self._check_frames(n_samples)
        arr = (C.c_void_p * self.S)(*[r._h for r in rings])
        L = load_library()
        return self._tick(lambda o, a, b, c: L.af_session_push_rings(self._h, arr, n_samples, o, a, b, c))

    def push_streams(self, xs, end=None) -> dict:
        """One tick in which stream k pushes xs[k] (1-D interleaved samples, any whole number of frames, 0 included); end[k]
        ends stream k after them (BatchResampler::flush), its next push starts afresh.  Returns per-stream lists."""
        buf, counts = stream_rows(xs, self.S, self.stream_channels(), np.int16 if self.fmt == AF_FMT_I16 else np.float32)
        e = end_flags(end, self.S)
        L = load_library()
        u32p = C.POINTER(C.c_uint32)
        return self._tick_streams(lambda o, a, b, c: L.af_session_push_streams(
            self._h, buf.ctypes.data, buf.shape[1], counts.ctypes.data_as(u32p),
            e.ctypes.data_as(C.POINTER(C.c_uint8)) if e is not None else None, AF_MEM_HOST, o, a, b, c))

    def reset_streams(self, ids):
        """Streams `ids` start afresh at their next push, without a flush; the others are untouched."""
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1)
        _check(load_library().af_session_reset_streams(self._h, a.ctypes.data_as(C.POINTER(C.c_uint32)), a.size))

    def restart_streams(self, ids, format_ids):
        """Streams `ids` start afresh at their next push in formats[format_ids[i]] (reset_streams plus a new format)."""
        a = np.ascontiguousarray(ids, dtype=np.int64).reshape(-1)
        f = np.ascontiguousarray(format_ids, dtype=np.int64).reshape(-1)
        if a.size != f.size:
            raise ValueError(f"{a.size} streams and {f.size} formats")
        if a.size and (a.min() < 0 or a.max() >= self.S):
            raise ValueError(f"stream index out of range ({self.S} streams)")
        if f.size and (f.min() < 0 or f.max() >= len(self.format_list)):
            raise ValueError(f"format index out of range ({len(self.format_list)} formats)")
        a32, f32 = a.astype(np.uint32), f.astype(np.uint32)
        u32p = C.POINTER(C.c_uint32)
        _check(load_library().af_session_restart_streams(self._h, a32.ctypes.data_as(u32p), f32.ctypes.data_as(u32p), a.size))
        self.stream_format[a32] = f32

    def set_vad_configs(self, ids, cfgs):
        """Stream ids[i] decides every frame completed from the next push on under cfgs[i] (the last entry wins for a
        stream listed twice); the detector keeps its state.  The configuration stays with the slot across resets,
        restarts and ends."""
        if not self.pipe.cfg.vad_enable:
            raise ValueError("the pipeline runs no VAD (vad_enable == 0)")
        a = np.ascontiguousarray(ids, dtype=np.int64).reshape(-1)
        cfgs = list(cfgs)
        if a.size != len(cfgs):
            raise ValueError(f"{a.size} streams and {len(cfgs)} configs")
        if a.size and (a.min() < 0 or a.max() >= self.S):
            raise ValueError(f"stream index out of range ({self.S} streams)")
        arr = _vad_config_array(cfgs)
        a32 = a.astype(np.uint32)
        _check(load_library().af_session_set_vad_configs(self._h, a32.ctypes.data_as(C.POINTER(C.c_uint32)), arr, a.size))

    def push_rings_available(self, rings, max_samples: int, end=None) -> dict:
        """AudioCapturer::read_frame(max) for every stream: min(max_samples, available) whole frames from each ring."""
        if len(rings) != self.S:
            raise ValueError(f"{len(rings)} rings for {self.S} streams")
        e = end_flags(end, self.S)
        arr = (C.c_void_p * self.S)(*[r._h for r in rings])
        L = load_library()
        return self._tick_streams(lambda o, a, b, c: L.af_session_push_rings_available(
            self._h, arr, max_samples, e.ctypes.data_as(C.POINTER(C.c_uint8)) if e is not None else None, o, a, b, c))

    def enable_wire(self, gate: bool, pcm16: bool = True, base64: bool = True, mem: int = AF_MEM_HOST):
        """Per-tick wire payloads (WebSocketClient::send_audio, websocket.rs:244-254); gate: speech frames only.
        gate=None switches the output off."""
        L = load_library()
        if gate is None:
            _check(L.af_session_enable_wire(self._h, None))
            self.wire_mem = None
            return
        cfg = WireConfigC(int(gate), int(pcm16), int(base64), mem)
        _check(L.af_session_enable_wire(self._h, C.byref(cfg)))
        self.wire_mem = mem

    def wire(self) -> dict:
        """The payloads of the last push: {"first_frame", "first_frames" (uint64[n_streams]: each stream's first completed
        frame in its own frame sequence), "streams": [per stream {pcm16: int16[n], base64: bytes, started,
        ended, in_speech, continued, n_samples, n_chars}]}.  With AF_MEM_DEVICE rows, pcm16 / base64 are None and the device
        rows are reported as "pcm16_ptr", "pcm16_stride" (elements), "base64_ptr", "base64_stride" (bytes)."""
        p, ps, b, bs, ff = C.c_void_p(), C.c_uint64(0), C.c_void_p(), C.c_uint64(0), C.c_uint64(0)
        ticks = (WireTickC * self.S)()
        _check(load_library().af_session_wire(self._h, C.byref(p), C.byref(ps), C.byref(b), C.byref(bs), ticks, C.byref(ff)))
        host = self.wire_mem == AF_MEM_HOST
        streams = []
        for k, t in enumerate(ticks):
            r = {"started": int(t.started), "ended": int(t.ended), "in_speech": bool(t.in_speech), "continued": int(t.continued),
                 "n_samples": int(t.n_samples), "n_chars": int(t.n_chars), "pcm16": None, "base64": None}
            if host and p.value:
                r["pcm16"] = np.ctypeslib.as_array((C.c_int16 * t.n_samples).from_address(p.value + 2 * k * ps.value)).copy() \
                    if t.n_samples else np.zeros(0, np.int16)
            if host and b.value:
                r["base64"] = C.string_at(b.value + k * bs.value, t.n_chars)
            streams.append(r)
        ffs = np.zeros(self.S, np.uint64)
        _check(load_library().af_session_wire_first_frames(self._h, ffs.ctypes.data_as(C.POINTER(C.c_uint64))))
        out = {"first_frame": int(ff.value), "first_frames": ffs, "streams": streams}
        if not host:
            out.update(pcm16_ptr=p.value, pcm16_stride=int(ps.value), base64_ptr=b.value, base64_stride=int(bs.value))
        return out


# ---------------------------------------------------------------------------------------------
# RingBuffer (capture.rs:84-161): the capture hand-off, same method names and semantics
# ---------------------------------------------------------------------------------------------
AF_RING_EMPTY = -1


class RingBuffer:
    def __init__(self, capacity_samples: int):
        h = C.c_void_p()
        _check(load_library().af_ring_create(capacity_samples, C.byref(h)))
        self._h = h
        self.capacity = int(load_library().af_ring_capacity(h))

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.af_ring_destroy(self._h)
            self._h = None

    def write(self, data) -> int:
        a = np.ascontiguousarray(data, dtype=np.float32)
        return int(load_library().af_ring_write(self._h, a.ctypes.data_as(C.POINTER(C.c_float)), a.size))

    def read(self, size: int):
        """None when nothing is available, else an array of min(size, available) samples."""
        out = np.empty(max(size, 1), np.float32)
        n = C.c_size_t(0)
        rc = load_library().af_ring_read(self._h, out.ctypes.data_as(C.POINTER(C.c_float)), size, C.byref(n))
        if rc == AF_RING_EMPTY:
            return None
        _check(rc)
        return out[:n.value].copy()

    def available(self) -> int:
        return int(load_library().af_ring_available(self._h))

    def clear(self):
        load_library().af_ring_clear(self._h)
