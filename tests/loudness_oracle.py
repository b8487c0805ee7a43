"""Test-side binding of tests/loudness_oracle.c: the CPU restatement of the loudness normalization (DESIGN.md 3.6).
Only tests/ and tools/ import this."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "loudness_oracle.c")
SO = os.path.join(HERE, "libctts_loudness_oracle.so")

K_MAX = 8000
UNITY = 65536


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
        d4 = [C.c_void_p] * 4
        L.ctts_oracle_loudness_filter.argtypes = [C.c_uint32] + d4
        L.ctts_oracle_loudness.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        L.ctts_oracle_loudness.restype = C.c_double
        L.ctts_oracle_loudness_table.argtypes = [C.c_int]
        L.ctts_oracle_loudness_table.restype = C.c_uint32
        L.ctts_oracle_loudness_ceiling.argtypes = [C.c_float]
        L.ctts_oracle_loudness_ceiling.restype = C.c_uint32
        L.ctts_oracle_loudness_gain.argtypes = [C.c_double, C.c_float, C.c_float, C.c_uint32]
        L.ctts_oracle_loudness_gain.restype = C.c_uint32
        L.ctts_oracle_loudness_normalize.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_float, C.c_float, C.c_void_p,
                                                     C.POINTER(C.c_double)]
        L.ctts_oracle_loudness_normalize.restype = C.c_uint32
        _lib = L
    return _lib


def filter_coeffs(fs: int) -> tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """(shelf b, shelf a, high-pass b, high-pass a), three each."""
    v = [np.zeros(3) for _ in range(4)]
    lib().ctts_oracle_loudness_filter(fs, *[a.ctypes.data for a in v])
    return tuple(v)


def lufs(x: np.ndarray, fs: int) -> float:
    x = np.ascontiguousarray(x, dtype=np.int16)
    return float(lib().ctts_oracle_loudness(x.ctypes.data, len(x), fs))


def table() -> np.ndarray:
    return np.array([lib().ctts_oracle_loudness_table(k) for k in range(-K_MAX, K_MAX + 1)], np.uint32)


def ceiling(c: float) -> int:
    return int(lib().ctts_oracle_loudness_ceiling(c))


def gain(L: float, target: float, ceiling_dbfs: float, peak: int) -> int:
    return int(lib().ctts_oracle_loudness_gain(L, target, ceiling_dbfs, peak))


def normalize(x: np.ndarray, fs: int, target: float, ceiling_dbfs: float) -> tuple[np.ndarray, float, int]:
    """(y, L, G) of one utterance."""
    x = np.ascontiguousarray(x, dtype=np.int16)
    y = np.zeros(max(len(x), 1), np.int16)
    L = C.c_double()
    G = lib().ctts_oracle_loudness_normalize(x.ctypes.data, len(x), fs, target, ceiling_dbfs, y.ctypes.data, C.byref(L))
    return y[:len(x)], float(L.value), int(G)


def near_tie(L: float, target: float) -> bool:
    """100 (T - L) within 1e-4 of a half-integer: the one case where the device's k may legitimately differ."""
    if not np.isfinite(L):
        return False
    v = 100.0 * (float(np.float32(target)) - L)
    return abs((v - 0.5) - np.round(v - 0.5)) < 1e-4
