"""ctypes binding of libctts_b200.so (include/ctts_b200.h): texts -> PCM, the text front end's planner
threads pipelined into a device session.  Product path: no CPU fallback for anything that touches samples."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build
from . import front as _front
from . import gpu as _gpu


class Options(C.Structure):
    _fields_ = [("piece_utts", C.c_uint32), ("threads", C.c_uint32), ("on_piece", C.c_void_p), ("user", C.c_void_p),
                ("cache", C.c_void_p)]


class Timing(C.Structure):
    _fields_ = [("first_plan_s", C.c_double), ("all_plans_s", C.c_double), ("all_submitted_s", C.c_double),
                ("done_s", C.c_double), ("wait_for_plans_s", C.c_double), ("pieces", C.c_uint32), ("reserved", C.c_uint32)]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _front.lib()          # the two libraries it is linked against, from the same directory
        _gpu.lib()
        path = _build.build_pipeline()
        if not os.path.exists(path):
            raise RuntimeError("libctts_b200.so is missing")
        L = C.CDLL(path)
        vp = C.c_void_p
        L.ctts_b200_synth_texts.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp, vp,
                                            C.POINTER(C.c_uint64), C.POINTER(Options), C.POINTER(Timing)]
        L.ctts_b200_capacity_hint.argtypes = [vp, vp, vp, C.c_uint32]
        L.ctts_b200_capacity_hint.restype = C.c_uint64
        L.ctts_b200_capacity_hint_rate.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint32]
        L.ctts_b200_capacity_hint_rate.restype = C.c_uint64
        L.ctts_b200_synth_texts_flac.argtypes = [vp, vp, vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp, vp, vp,
                                                 C.POINTER(C.c_uint64), C.POINTER(Options), C.POINTER(Timing)]
        L.ctts_b200_capacity_hint_flac.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint32]
        L.ctts_b200_capacity_hint_flac.restype = C.c_uint64
        L.ctts_b200_synth_texts_g711.argtypes = [vp, vp, C.c_int, vp, vp, C.c_uint32, vp, C.c_uint64, vp, vp, vp,
                                                 C.POINTER(C.c_uint64), C.POINTER(Options), C.POINTER(Timing)]
        L.ctts_b200_plan_cache_create.argtypes = [C.c_size_t]
        L.ctts_b200_plan_cache_create.restype = vp
        L.ctts_b200_plan_cache_destroy.argtypes = [vp]
        L.ctts_b200_plan_cache_destroy.restype = None
        L.ctts_b200_plan_cache_stats.argtypes = [vp] + [C.POINTER(C.c_uint64)] * 4
        L.ctts_b200_plan_cache_stats.restype = None
        _lib = L
    return _lib


class PlanCache:
    """ctts_b200_plan_cache: plans by text, for callers that see the same sentences again."""

    def __init__(self, max_bytes: int = 256 << 20):
        self._h = lib().ctts_b200_plan_cache_create(max_bytes)
        if not self._h:
            raise MemoryError("ctts_b200_plan_cache_create")

    def stats(self) -> dict:
        v = [C.c_uint64() for _ in range(4)]
        lib().ctts_b200_plan_cache_stats(self._h, *[C.byref(x) for x in v])
        return dict(zip(("hits", "misses", "entries", "bytes"), (int(x.value) for x in v)))

    def close(self) -> None:
        if self._h:
            lib().ctts_b200_plan_cache_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TextBatch:
    """N texts as the C strings the entry point takes (built once; what a C caller already has)."""

    def __init__(self, texts: list[str], speeds=None):
        self.n = len(texts)
        self._enc = [t.encode("utf-8") for t in texts]
        self.ptrs = (C.c_char_p * max(self.n, 1))(*self._enc)
        self.speeds = None if speeds is None else np.ascontiguousarray(speeds, dtype=np.float32)
        assert self.speeds is None or self.speeds.shape == (self.n,)

    @property
    def speeds_ptr(self):
        return None if self.speeds is None else self.speeds.ctypes.data


def capacity_hint(front, batch: TextBatch, rate: int = 22050) -> int:
    """Samples at output rate `rate` that are always enough for the batch (ctts_b200_capacity_hint_rate)."""
    if rate == 22050:
        return int(lib().ctts_b200_capacity_hint(front._h, batch.ptrs, batch.speeds_ptr, batch.n))
    return int(lib().ctts_b200_capacity_hint_rate(front._h, batch.ptrs, batch.speeds_ptr, batch.n, rate))


def synth_texts(front, gpu, batch: TextBatch, pcm_out: np.ndarray, piece_utts: int = 0, threads: int = 0,
                want_stats: bool = False, cache: PlanCache | None = None):
    """ctts_b200_synth_texts.  Returns (offsets[n], counts[n], samples_used, Timing[, stats])."""
    assert pcm_out.dtype == np.int16 and pcm_out.flags["C_CONTIGUOUS"]
    n = batch.n
    off = np.zeros(max(n, 1), dtype=np.uint64)
    cnt = np.zeros(max(n, 1), dtype=np.uint32)
    stats = np.zeros(2 * max(n, 1), dtype=np.uint32) if want_stats else None
    used = C.c_uint64()
    opt = Options(piece_utts, threads, None, None, cache._h if cache is not None else None)
    tm = Timing()
    rc = lib().ctts_b200_synth_texts(front._h, gpu._h, batch.ptrs, batch.speeds_ptr, n, pcm_out.ctypes.data,
                                     pcm_out.size, off.ctypes.data, cnt.ctypes.data,
                                     stats.ctypes.data if want_stats else None, C.byref(used), C.byref(opt), C.byref(tm))
    if rc != 0:
        msg = _gpu.lib().ctts_gpu_last_error(gpu._h)
        raise _gpu.GpuError(f"ctts_b200_synth_texts: {rc}: {msg.decode(errors='replace') if msg else ''}")
    res = (off[:n], cnt[:n], int(used.value), tm)
    return res + (stats[:2 * n].reshape(n, 2),) if want_stats else res


def capacity_hint_flac(front, batch: TextBatch, rate: int = 22050) -> int:
    """Bytes that are always enough for synth_texts_flac at output rate `rate` (ctts_b200_capacity_hint_flac)."""
    return int(lib().ctts_b200_capacity_hint_flac(front._h, batch.ptrs, batch.speeds_ptr, batch.n, rate))


def synth_texts_flac(front, gpu, batch: TextBatch, out: np.ndarray, piece_utts: int = 0, threads: int = 0,
                     cache: PlanCache | None = None):
    """ctts_b200_synth_texts_flac: one .flac file per utterance in the uint8 buffer `out`.
    Returns (byte offsets[n], file bytes[n], sample counts[n], bytes_used, Timing)."""
    assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
    n = batch.n
    off = np.zeros(max(n, 1), dtype=np.uint64)
    nbytes = np.zeros(max(n, 1), dtype=np.uint32)
    cnt = np.zeros(max(n, 1), dtype=np.uint32)
    used = C.c_uint64()
    opt = Options(piece_utts, threads, None, None, cache._h if cache is not None else None)
    tm = Timing()
    rc = lib().ctts_b200_synth_texts_flac(front._h, gpu._h, batch.ptrs, batch.speeds_ptr, n, out.ctypes.data, out.size,
                                          off.ctypes.data, nbytes.ctypes.data, cnt.ctypes.data, None, C.byref(used),
                                          C.byref(opt), C.byref(tm))
    if rc != 0:
        msg = _gpu.lib().ctts_gpu_last_error(gpu._h)
        raise _gpu.GpuError(f"ctts_b200_synth_texts_flac: {rc}: {msg.decode(errors='replace') if msg else ''}")
    return off[:n], nbytes[:n], cnt[:n], int(used.value), tm


def synth_texts_g711(front, gpu, batch: TextBatch, law: int, out: np.ndarray, piece_utts: int = 0, threads: int = 0,
                     cache: PlanCache | None = None):
    """ctts_b200_synth_texts_g711: one G.711 byte of `law` (gpu.G711_ULAW or gpu.G711_ALAW) per sample in the uint8
    buffer `out`, in the packed layout; capacity_hint(front, batch, rate) bytes are always enough.
    Returns (byte offsets[n], sample counts[n], bytes_used, Timing)."""
    assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
    n = batch.n
    off = np.zeros(max(n, 1), dtype=np.uint64)
    cnt = np.zeros(max(n, 1), dtype=np.uint32)
    used = C.c_uint64()
    opt = Options(piece_utts, threads, None, None, cache._h if cache is not None else None)
    tm = Timing()
    rc = lib().ctts_b200_synth_texts_g711(front._h, gpu._h, law, batch.ptrs, batch.speeds_ptr, n, out.ctypes.data, out.size,
                                          off.ctypes.data, cnt.ctypes.data, None, C.byref(used), C.byref(opt), C.byref(tm))
    if rc != 0:
        msg = _gpu.lib().ctts_gpu_last_error(gpu._h)
        raise _gpu.GpuError(f"ctts_b200_synth_texts_g711: {rc}: {msg.decode(errors='replace') if msg else ''}")
    return off[:n], cnt[:n], int(used.value), tm
