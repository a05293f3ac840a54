"""ctypes front-end of oracle/polyphase.c: the CPU definition of af_batch_set_resampler(AF_RESAMPLE_POLYPHASE).

TEST INFRASTRUCTURE ONLY, like oracle.py.  The shared library is compiled on first use into a per-user directory under
the system's temporary directory, named after a hash of the source, so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "polyphase.c")
_CFLAGS = ["-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-fvisibility=hidden", "-Wall", "-Wextra", "-std=c11"]
_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    with open(_SRC, "rb") as f:
        tag = hashlib.sha256(f.read() + " ".join(_CFLAGS).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"audioflow_oracle_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    path = os.path.join(d, f"libpolyphase_{tag}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), *_CFLAGS, "-shared", "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, path)                      # atomic: concurrent test processes never load a half-written file
    L = C.CDLL(path)
    fp = C.POINTER(C.c_float)
    L.orc_resample_polyphase.restype = None
    L.orc_resample_polyphase.argtypes = [fp, C.c_size_t, C.c_uint32, C.c_uint32, fp, C.c_size_t, C.c_size_t, fp]
    _lib = L
    return L


def resample_polyphase(mono, p: int, q: int, h, n_out: int) -> np.ndarray:
    """orc_resample_polyphase over a mono f32 signal, with the tap table h (2L + 1 taps) given."""
    m = np.ascontiguousarray(mono, dtype=np.float32)
    hh = np.ascontiguousarray(h, dtype=np.float32)
    y = np.empty(max(n_out, 1), np.float32)
    fp = C.POINTER(C.c_float)
    lib().orc_resample_polyphase(m.ctypes.data_as(fp), len(m), p, q, hh.ctypes.data_as(fp), len(hh), n_out,
                                 y.ctypes.data_as(fp))
    return y[:n_out]
