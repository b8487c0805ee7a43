"""Test-side binding of tests/true_peak_oracle.c: the CPU restatement of the true-peak ceiling of the loudness
normalization (DESIGN.md 3.6).  L comes from loudness_oracle.  Only tests/ and tools/ import this."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

import loudness_oracle as LO

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "true_peak_oracle.c")
SO = os.path.join(HERE, "libctts_true_peak_oracle.so")


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
        L.ctts_oracle_true_peak_taps.argtypes = [C.c_void_p]
        L.ctts_oracle_true_peak_taps.restype = None
        L.ctts_oracle_true_peak.argtypes = [C.c_void_p, C.c_uint64]
        L.ctts_oracle_true_peak.restype = C.c_float
        L.ctts_oracle_true_peak_gain.argtypes = [C.c_double, C.c_float, C.c_float, C.c_float]
        L.ctts_oracle_true_peak_gain.restype = C.c_uint32
        L.ctts_oracle_true_peak_apply.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p]
        L.ctts_oracle_true_peak_apply.restype = None
        _lib = L
    return _lib


def taps() -> np.ndarray:
    """The 49 interpolator taps as float32, computed by the oracle from the formula."""
    h = np.zeros(49, np.float32)
    lib().ctts_oracle_true_peak_taps(h.ctypes.data)
    return h


def true_peak(x: np.ndarray) -> float:
    """P of one utterance (a float32 value, as a Python float)."""
    x = np.ascontiguousarray(x, dtype=np.int16)
    return float(lib().ctts_oracle_true_peak(x.ctypes.data, len(x)))


def gain(L: float, target: float, ceiling_dbtp: float, peak: float) -> int:
    return int(lib().ctts_oracle_true_peak_gain(L, target, ceiling_dbtp, peak))


def normalize(x: np.ndarray, fs: int, target: float, ceiling_dbtp: float) -> tuple[np.ndarray, float, int, float]:
    """(y, L, G, P) of one utterance under a true-peak ceiling."""
    x = np.ascontiguousarray(x, dtype=np.int16)
    P = true_peak(x)
    L = LO.lufs(x, fs)
    G = gain(L, target, ceiling_dbtp, P)
    y = np.zeros(max(len(x), 1), np.int16)
    lib().ctts_oracle_true_peak_apply(x.ctypes.data, len(x), G, y.ctypes.data)
    return y[:len(x)], L, G, P
