"""Test-side binding of tests/resample_oracle.c: the CPU restatement of the output-rate conversion
(DESIGN.md 3.4).  Only tests/ and tools/ import this."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "resample_oracle.c")
SO = os.path.join(HERE, "libctts_resample_oracle.so")

NATIVE = 22050
# the rates the issue of the feature names; every integer rate in [8000, 48000] with max(L, M) <= 1024 is accepted
COMMON_RATES = (8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000)
H_ZERO_CROSSINGS = 40


def build() -> str:
    if not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
        cc = shutil.which("gcc") or "cc"
        subprocess.run([cc, "-O2", "-std=c99", "-ffp-contract=off", "-Wall", "-Wextra", "-fPIC", "-shared", "-o", SO, SRC, "-lm"],
                       check=True)
    return SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.ctts_oracle_resample_ratio.argtypes = [C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.ctts_oracle_resample_taps.argtypes = [C.c_uint32, C.c_void_p, C.c_size_t]
        L.ctts_oracle_resample_taps.restype = C.c_size_t
        L.ctts_oracle_resample_count.argtypes = [C.c_uint32, C.c_uint64]
        L.ctts_oracle_resample_count.restype = C.c_uint64
        L.ctts_oracle_resample.argtypes = [C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]
        L.ctts_oracle_resample.restype = C.c_int64
        _lib = L
    return _lib


def ratio(hz: int) -> tuple[int, int] | None:
    """(L, M) of an accepted rate, None otherwise."""
    a, b = C.c_uint32(), C.c_uint32()
    if lib().ctts_oracle_resample_ratio(hz, C.byref(a), C.byref(b)):
        return None
    return int(a.value), int(b.value)


def taps(hz: int) -> np.ndarray:
    L, M = ratio(hz)
    n = 2 * H_ZERO_CROSSINGS * max(L, M) + 1
    g = np.zeros(n, np.float32)
    assert lib().ctts_oracle_resample_taps(hz, g.ctypes.data, n) == n
    return g


def count(hz: int, n: int) -> int:
    return int(lib().ctts_oracle_resample_count(hz, n))


def resample(x: np.ndarray, hz: int) -> np.ndarray:
    """Native-rate int16 PCM -> int16 PCM at hz (22050: a copy)."""
    x = np.ascontiguousarray(x, dtype=np.int16)
    if hz == NATIVE:
        return x.copy()
    n_out = count(hz, len(x))
    y = np.zeros(max(n_out, 1), np.int16)
    got = lib().ctts_oracle_resample(hz, x.ctypes.data, len(x), y.ctypes.data)
    assert got == n_out
    return y[:n_out]
