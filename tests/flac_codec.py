"""Test-side bindings of the two FLAC programs that pin the format (DESIGN.md 3.5), built as separate libraries that
share no code: tests/flac_oracle.c (the encoder contract restated) and tests/flac_decode.c (an RFC 9639 decoder).
Only tests/ and tools/ import this."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = {"oracle": "flac_oracle.c", "decode": "flac_decode.c"}
BLOCK = 4096
FRAME_MAX = 16 + 1 + 2 * BLOCK + 2
INFO_FIELDS = ("min_blocksize", "max_blocksize", "min_framesize", "max_framesize", "sample_rate", "channels",
               "bits_per_sample", "total_samples", "md5_zero")
# per frame, what the decoder parsed (ctts_flac_decode_report); kind 0 CONSTANT, 1 VERBATIM, 2 FIXED, 3 LPC
REPORT_FIELDS = ("number", "blocksize", "header_bytes", "kind", "order", "po", "kmin", "kmax")
CONSTANT, VERBATIM, FIXED = 0, 1, 2


class DecodeError(ValueError):
    pass


def _so(name: str) -> str:
    return os.path.join(HERE, f"libctts_flac_{name}.so")


def build() -> list[str]:
    cc = shutil.which("gcc") or "cc"
    out = []
    for name, src in SOURCES.items():
        src, so = os.path.join(HERE, src), _so(name)
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
            subprocess.run([cc, "-O2", "-std=c99", "-Wall", "-Wextra", "-fPIC", "-shared", "-o", so, src], check=True)
        out.append(so)
    return out


_libs: dict = {}


def _lib(name: str) -> C.CDLL:
    if name not in _libs:
        build()
        L = C.CDLL(_so(name))
        if name == "oracle":
            L.ctts_flac_oracle_encode.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint64]
            L.ctts_flac_oracle_encode.restype = C.c_int64
        else:
            L.ctts_flac_decode.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]
            L.ctts_flac_decode.restype = C.c_int64
            L.ctts_flac_decode_report.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                                  C.c_uint64, C.POINTER(C.c_uint64)]
            L.ctts_flac_decode_report.restype = C.c_int64
        _libs[name] = L
    return _libs[name]


def bound(n: int) -> int:
    """The size bound of the contract, restated: 42 + ceil(n / 4096) * 8211."""
    return 42 + -(-n // BLOCK) * FRAME_MAX


def encode(x, hz: int) -> bytes:
    """The oracle encoder: int16 PCM -> the bytes of its .flac file."""
    x = np.ascontiguousarray(x, dtype=np.int16)
    cap = bound(len(x))
    buf = np.zeros(cap, np.uint8)
    got = _lib("oracle").ctts_flac_oracle_encode(x.ctypes.data, len(x), hz, buf.ctypes.data, cap)
    assert got >= 0, "oracle: buffer too small"
    return buf[:got].tobytes()


def decode(data: bytes, cap: int | None = None, report: bool = False):
    """The independent decoder: .flac bytes -> (int16 PCM, STREAMINFO fields); DecodeError for a malformed stream.
    With report, also a record array of the frames as parsed (REPORT_FIELDS), the decoder's witness of what the
    encoder chose."""
    src = np.frombuffer(data, np.uint8)
    if cap is None:   # STREAMINFO's total, when the header is there to read
        cap = int.from_bytes(data[21:26], "big") & ((1 << 36) - 1) if len(data) >= 26 else 0
        cap = max(cap, 1 << 16)
    out = np.zeros(max(cap, 1), np.int16)
    info = np.zeros(len(INFO_FIELDS), np.uint64)
    rep_cap = len(data) // 6 + 1 if report else 0   # a frame takes at least 6 bytes
    rep = np.zeros((max(rep_cap, 1), len(REPORT_FIELDS)), np.uint32)
    frames = C.c_uint64()
    got = _lib("decode").ctts_flac_decode_report(src.ctypes.data if len(src) else None, len(src), out.ctypes.data, cap,
                                                 info.ctypes.data, rep.ctypes.data if report else None, rep_cap,
                                                 C.byref(frames))
    if got < 0:
        raise DecodeError(f"flac_decode: error {got}")
    res = out[:got].copy(), dict(zip(INFO_FIELDS, (int(v) for v in info)))
    if not report:
        return res
    return res + (np.rec.fromarrays(list(rep[:frames.value].astype(np.int64).T), names=REPORT_FIELDS),)
