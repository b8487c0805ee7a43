"""ctypes binding of the C-ABI back end (include/ctts_gpu.h, libctts_gpu.so).

The product path: there is no CPU fallback.  If the CUDA library is missing or
no device is present every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import numpy as np

from . import _build
from .front import AssemblyParams, BatchPlan, CBatchPlan

ERR_CUDA, ERR_BOUNDS, ERR_DEVICE = -100, -101, -102
G711_ULAW, G711_ALAW = 1, 2   # CTTS_GPU_G711_ULAW, CTTS_GPU_G711_ALAW


class WsolaStats(C.Structure):
    _fields_ = [("frames", C.c_uint64), ("tier2_candidates", C.c_uint64), ("exact_evaluations", C.c_uint64),
                ("walked_utterances", C.c_uint64), ("walked_frames", C.c_uint64)]


class RunInfo(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint32), ("n_stretch", C.c_uint32),
        ("gather_samples", C.c_uint64), ("bound_samples", C.c_uint64),
        ("smem_bytes", C.c_uint32), ("window_samples", C.c_uint32),
        ("halo_samples", C.c_uint32), ("threads", C.c_uint32),
        ("n_tasks", C.c_uint32), ("n_global_tasks", C.c_uint32),
        ("ctas_per_sm", C.c_uint32), ("grid", C.c_uint32),
        ("n_canon_tasks", C.c_uint32), ("n_dedup_tasks", C.c_uint32), ("dedup_bound_samples", C.c_uint64),
        ("n_source_tasks", C.c_uint32), ("n_reuse_tasks", C.c_uint32), ("reuse_bound_samples", C.c_uint64),
    ]


_lib = None


def lib(build: bool = True) -> C.CDLL:
    """Loads libctts_gpu.so (building it in-tree with nvcc if the sources are newer)."""
    global _lib
    if _lib is None:
        path = _build.build_gpu() if build else _build.GPU_SO
        path = os.environ.get("CTTS_GPU_LIB", path)   # development: A/B a differently built library
        if not os.path.exists(path):
            raise RuntimeError("libctts_gpu.so is missing: the CUDA back end has no CPU fallback")
        L = C.CDLL(path)
        vp, u64p, u32p = C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
        L.ctts_gpu_init.argtypes = [C.POINTER(vp), vp, C.c_size_t, C.c_int]
        L.ctts_gpu_free.argtypes = [vp]
        L.ctts_gpu_free.restype = None
        L.ctts_gpu_set_stream.argtypes = [vp, vp]
        L.ctts_gpu_set_output_rate.argtypes = [vp, C.c_uint32]
        L.ctts_gpu_set_loudness.argtypes = [vp, C.c_float, C.c_float]
        L.ctts_gpu_plan_read_loudness.argtypes = [vp, vp, vp, vp]
        L.ctts_gpu_set_loudness_true_peak.argtypes = [vp, C.c_float, C.c_float]
        L.ctts_gpu_plan_read_true_peak.argtypes = [vp, vp, vp]
        L.ctts_gpu_last_error.argtypes = [vp]
        L.ctts_gpu_last_error.restype = C.c_char_p
        L.ctts_gpu_plan_bounds.argtypes = [vp, C.POINTER(CBatchPlan), vp]
        L.ctts_gpu_synth_batch.argtypes = [vp, C.POINTER(CBatchPlan), C.POINTER(AssemblyParams), vp, vp, vp]
        L.ctts_gpu_plan_create.argtypes = [vp, C.POINTER(CBatchPlan), C.POINTER(AssemblyParams), vp, C.POINTER(vp)]
        L.ctts_gpu_plan_destroy.argtypes = [vp]
        L.ctts_gpu_plan_destroy.restype = None
        L.ctts_gpu_plan_out_samples.argtypes = [vp]
        L.ctts_gpu_plan_out_samples.restype = C.c_uint64
        L.ctts_gpu_plan_out_offsets.argtypes = [vp, vp]
        L.ctts_gpu_plan_run.argtypes = [vp, vp, vp]
        L.ctts_gpu_plan_read_counts.argtypes = [vp, vp, vp]
        L.ctts_gpu_plan_read_pcm.argtypes = [vp, vp, vp, C.c_uint64, C.c_uint64]
        L.ctts_gpu_plan_read_pre.argtypes = [vp, vp, C.c_uint32, vp, C.c_uint64, u64p]
        L.ctts_gpu_plan_info.argtypes = [vp, C.POINTER(RunInfo)]
        L.ctts_gpu_plan_wsola_stats.argtypes = [vp, vp, C.POINTER(WsolaStats)]
        L.ctts_gpu_session_begin.argtypes = [vp, C.POINTER(AssemblyParams), vp, C.c_uint64, vp, vp, C.POINTER(vp)]
        L.ctts_gpu_session_submit.argtypes = [vp, C.POINTER(CBatchPlan), vp, vp]
        L.ctts_gpu_session_end.argtypes = [vp, u64p]
        L.ctts_gpu_session_begin_flac.argtypes = [vp, C.POINTER(AssemblyParams), vp, C.c_uint64, vp, vp, C.POINTER(vp)]
        L.ctts_gpu_session_submit_flac.argtypes = [vp, C.POINTER(CBatchPlan), vp, vp, vp]
        L.ctts_gpu_flac_bound.argtypes = [C.c_uint64]
        L.ctts_gpu_flac_bound.restype = C.c_uint64
        L.ctts_gpu_session_begin_g711.argtypes = [vp, C.POINTER(AssemblyParams), C.c_int, vp, C.c_uint64, vp, vp, C.POINTER(vp)]
        L.ctts_gpu_session_submit_g711.argtypes = [vp, C.POINTER(CBatchPlan), vp, vp]
        L.ctts_gpu_synth_batch_packed.argtypes = [vp, C.POINTER(CBatchPlan), C.POINTER(AssemblyParams), vp, C.c_uint64, vp, vp, u64p]
        L.ctts_gpu_multi_synth_batch.argtypes = [C.POINTER(vp), C.c_uint32, C.POINTER(CBatchPlan), C.POINTER(AssemblyParams),
                                                 vp, vp, vp, vp]
        _lib = L
    return _lib


class GpuError(RuntimeError):
    pass


class ResidentPlan:
    """A plan uploaded to the device with its workspace (ctts_gpu_plan)."""

    def __init__(self, ctx: "GpuSynth", handle, n_utts: int):
        self._ctx = ctx
        self._h = handle
        self.n_utts = n_utts

    def close(self) -> None:
        # a plan points into its context, so it is never destroyed after ctts_gpu_free.  GpuSynth.close destroys
        # the plans it still knows first.  When the garbage collector frees a context and its plans together
        # (a reference cycle) it clears the weak references before any finalizer runs, the context goes first
        # and the plan's device memory is left allocated until the process ends: a leak, not a crash.
        if self._h:
            if self._ctx._h:
                lib().ctts_gpu_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def out_samples(self) -> int:
        return int(lib().ctts_gpu_plan_out_samples(self._h))

    def out_offsets(self) -> np.ndarray:
        off = np.zeros(self.n_utts + 1, dtype=np.uint64)
        self._ctx._check(lib().ctts_gpu_plan_out_offsets(self._h, off.ctypes.data))
        return off

    def info(self) -> RunInfo:
        r = RunInfo()
        self._ctx._check(lib().ctts_gpu_plan_info(self._h, C.byref(r)))
        return r

    def run(self, d_out_ptr: int | None = None) -> None:
        """Enqueue the batch on the context stream (asynchronous)."""
        self._ctx._check(lib().ctts_gpu_plan_run(self._ctx._h, self._h, d_out_ptr))

    def counts(self) -> np.ndarray:
        c = np.zeros(max(self.n_utts, 1), dtype=np.uint32)
        self._ctx._check(lib().ctts_gpu_plan_read_counts(self._ctx._h, self._h, c.ctypes.data))
        return c[:self.n_utts]

    def read_pcm(self, first: int, n: int) -> np.ndarray:
        out = np.zeros(max(n, 1), dtype=np.int16)
        self._ctx._check(lib().ctts_gpu_plan_read_pcm(self._ctx._h, self._h, out.ctypes.data, first, n))
        return out[:n]

    def loudness(self) -> tuple[np.ndarray, np.ndarray]:
        """After a run of a plan created with loudness normalization on (ctts_gpu_plan_read_loudness): every
        utterance's integrated loudness in LUFS (-inf when undefined) and the Q16 gain applied to it."""
        lufs = np.zeros(max(self.n_utts, 1), dtype=np.float64)
        gain = np.zeros(max(self.n_utts, 1), dtype=np.uint32)
        self._ctx._check(lib().ctts_gpu_plan_read_loudness(self._ctx._h, self._h, lufs.ctypes.data, gain.ctypes.data))
        return lufs[:self.n_utts], gain[:self.n_utts]

    def true_peak(self) -> np.ndarray:
        """After a run of a plan created under a true-peak ceiling (ctts_gpu_plan_read_true_peak): every utterance's
        true peak P (4x oversampled, int16 units, float32) before the gain."""
        peak = np.zeros(max(self.n_utts, 1), dtype=np.float32)
        self._ctx._check(lib().ctts_gpu_plan_read_true_peak(self._ctx._h, self._h, peak.ctypes.data))
        return peak[:self.n_utts]

    def read_pre(self, u: int, cap: int) -> np.ndarray:
        out = np.zeros(max(cap, 1), dtype=np.int16)
        n = C.c_uint64()
        self._ctx._check(lib().ctts_gpu_plan_read_pre(self._ctx._h, self._h, u, out.ctypes.data, cap, C.byref(n)))
        return out[:min(int(n.value), cap)]

    def wsola_stats(self) -> WsolaStats:
        """How the WSOLA frame chain of the last run was resolved (ctts_gpu_wsola_stats)."""
        st = WsolaStats()
        self._ctx._check(lib().ctts_gpu_plan_wsola_stats(self._ctx._h, self._h, C.byref(st)))
        return st

    def utterances(self) -> list[np.ndarray]:
        """Convenience for tests: per-utterance PCM read back from the plan-owned buffer."""
        cnt = self.counts()
        off = self.out_offsets()
        return [self.read_pcm(int(off[u]), int(cnt[u])) for u in range(self.n_utts)]


class GpuSynth:
    """One context per GPU: HBM-resident PCM pool + tables (ctts_gpu_ctx)."""

    def __init__(self, voice_db: bytes, device: int = 0):
        L = lib()
        h = C.c_void_p()
        buf = (C.c_char * len(voice_db)).from_buffer_copy(voice_db)
        rc = L.ctts_gpu_init(C.byref(h), C.addressof(buf), len(voice_db), device)
        if rc != 0:
            why = L.ctts_gpu_last_error(None)
            raise GpuError(f"ctts_gpu_init failed: {rc}: {why.decode(errors='replace') if why else ''}")
        self._h = h
        self.device = device
        self._plans = weakref.WeakSet()

    def close(self) -> None:
        if self._h:
            for p in list(self._plans):
                p.close()
            lib().ctts_gpu_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int) -> None:
        if rc != 0:
            msg = lib().ctts_gpu_last_error(self._h)
            raise GpuError(f"ctts_gpu error {rc}: {msg.decode(errors='replace') if msg else ''}")

    def set_stream(self, cuda_stream_ptr: int | None) -> None:
        self._check(lib().ctts_gpu_set_stream(self._h, cuda_stream_ptr))

    def set_output_rate(self, hz: int) -> None:
        """ctts_gpu_set_output_rate: every later call of this context delivers PCM at `hz` (8000..48000, see
        ctts_gpu.h for the accepted rates; 22050 is the voice's own), and every count, offset and bound is in
        samples of that rate.  Plans created before keep their rate."""
        self._check(lib().ctts_gpu_set_output_rate(self._h, int(hz)))

    def set_loudness(self, target_lufs: float, ceiling_dbfs: float = -1.0, true_peak: bool = False) -> None:
        """ctts_gpu_set_loudness: every later call of this context normalizes each utterance to target_lufs LUFS
        (ITU-R BS.1770-4, in [-60, -5]) without letting its sample peak pass ceiling_dbfs dBFS (in [-20, 0]).
        true_peak=True (ctts_gpu_set_loudness_true_peak): the ceiling is in dBTP and holds the 4x oversampled peak.
        target_lufs == 0 turns it off.  Plans created before keep their setting."""
        f = lib().ctts_gpu_set_loudness_true_peak if true_peak else lib().ctts_gpu_set_loudness
        self._check(f(self._h, float(target_lufs), float(ceiling_dbfs)))

    def bounds(self, plan: BatchPlan) -> np.ndarray:
        b = np.zeros(max(plan.n_utts, 1), dtype=np.uint64)
        cp = plan.as_c()
        self._check(lib().ctts_gpu_plan_bounds(self._h, C.byref(cp), b.ctypes.data))
        return b[:plan.n_utts]

    def layout(self, plan: BatchPlan) -> np.ndarray:
        """16-byte aligned packed slot offsets (n_utts+1) sized by the bounds."""
        b = self.bounds(plan)
        off = np.zeros(plan.n_utts + 1, dtype=np.uint64)
        off[1:] = np.cumsum(((b + np.uint64(7)) // np.uint64(8)) * np.uint64(8) + np.uint64(8))
        return off

    def synth_batch(self, plan: BatchPlan, params: AssemblyParams, pcm_out: np.ndarray | None = None,
                    out_offsets: np.ndarray | None = None):
        """The drop-in call: host plan in, host PCM out (ctts_gpu_synth_batch). Returns (pcm, offsets, counts)."""
        if out_offsets is None:
            out_offsets = self.layout(plan)
        out_offsets = np.ascontiguousarray(out_offsets, dtype=np.uint64)
        total = int(out_offsets[-1])
        if pcm_out is None:
            pcm_out = np.empty(max(total, 1), dtype=np.int16)
        assert pcm_out.dtype == np.int16 and pcm_out.size >= total and pcm_out.flags["C_CONTIGUOUS"]
        counts = np.zeros(max(plan.n_utts, 1), dtype=np.uint32)
        cp = plan.as_c()
        self._check(lib().ctts_gpu_synth_batch(self._h, C.byref(cp), C.byref(params), pcm_out.ctypes.data,
                                               out_offsets.ctypes.data, counts.ctypes.data))
        return pcm_out, out_offsets, counts[:plan.n_utts]

    def synth_batch_packed(self, plan: BatchPlan, params: AssemblyParams, pcm_out: np.ndarray):
        """ctts_gpu_synth_batch_packed: library-chosen packed layout. Returns (offsets[n], counts[n], samples_used)."""
        assert pcm_out.dtype == np.int16 and pcm_out.flags["C_CONTIGUOUS"]
        n = plan.n_utts
        off = np.zeros(max(n, 1), dtype=np.uint64)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        used = C.c_uint64()
        cp = plan.as_c()
        self._check(lib().ctts_gpu_synth_batch_packed(self._h, C.byref(cp), C.byref(params), pcm_out.ctypes.data, pcm_out.size,
                                                       off.ctypes.data, cnt.ctypes.data, C.byref(used)))
        return off[:n], cnt[:n], int(used.value)

    def synth_batch_stream(self, plan: BatchPlan, params: AssemblyParams, on_chunk, pcm_out: np.ndarray | None = None,
                           out_offsets: np.ndarray | None = None):
        """ctts_gpu_synth_batch_stream: on_chunk(pcm, offsets, counts, utt_begin, utt_end) is called, in utterance
        order, as soon as that range of utterances is in host memory.  Returns (pcm, offsets, counts)."""
        if out_offsets is None:
            out_offsets = self.layout(plan)
        out_offsets = np.ascontiguousarray(out_offsets, dtype=np.uint64)
        total = int(out_offsets[-1])
        if pcm_out is None:
            pcm_out = np.empty(max(total, 1), dtype=np.int16)
        assert pcm_out.dtype == np.int16 and pcm_out.size >= total and pcm_out.flags["C_CONTIGUOUS"]
        counts = np.zeros(max(plan.n_utts, 1), dtype=np.uint32)
        cp = plan.as_c()
        fn_t = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.c_uint32)
        cb = fn_t(lambda _user, b, e: on_chunk(pcm_out, out_offsets, counts, int(b), int(e)))
        L = lib()
        L.ctts_gpu_synth_batch_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, fn_t, C.c_void_p]
        self._check(L.ctts_gpu_synth_batch_stream(self._h, C.byref(cp), C.byref(params), pcm_out.ctypes.data,
                                                  out_offsets.ctypes.data, counts.ctypes.data, cb, None))
        return pcm_out, out_offsets, counts[:plan.n_utts]

    def synth_pieces(self, pieces: list[BatchPlan], params: AssemblyParams, pcm_out: np.ndarray):
        """A session fed with the given plans, one piece each (ctts_gpu_session_*).
        Returns (offsets, counts) over all utterances of all pieces, in order."""
        L = lib()
        h = C.c_void_p()
        self._check(L.ctts_gpu_session_begin(self._h, C.byref(params), pcm_out.ctypes.data, pcm_out.size, None, None, C.byref(h)))
        n = sum(p.n_utts for p in pieces)
        off = np.zeros(max(n, 1), dtype=np.uint64)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        at, rc = 0, 0
        for p in pieces:
            cp = p.as_c()
            rc = L.ctts_gpu_session_submit(h, C.byref(cp), off[at:].ctypes.data, cnt[at:].ctypes.data)
            if rc:
                break
            at += p.n_utts
        used = C.c_uint64()
        rc_end = L.ctts_gpu_session_end(h, C.byref(used))
        self._check(rc or rc_end)
        return off[:n], cnt[:n]

    def synth_pieces_flac(self, pieces: list[BatchPlan], params: AssemblyParams, out: np.ndarray):
        """A FLAC session fed with the given plans, one piece each (ctts_gpu_session_begin_flac / _submit_flac): every
        utterance becomes one .flac file in the uint8 buffer `out`.  Returns (byte offsets, file bytes, sample counts,
        bytes used) over all utterances of all pieces, in order."""
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
        L = lib()
        h = C.c_void_p()
        self._check(L.ctts_gpu_session_begin_flac(self._h, C.byref(params), out.ctypes.data, out.size, None, None, C.byref(h)))
        n = sum(p.n_utts for p in pieces)
        off = np.zeros(max(n, 1), dtype=np.uint64)
        nbytes = np.zeros(max(n, 1), dtype=np.uint32)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        at, rc = 0, 0
        for p in pieces:
            cp = p.as_c()
            rc = L.ctts_gpu_session_submit_flac(h, C.byref(cp), off[at:].ctypes.data, nbytes[at:].ctypes.data, cnt[at:].ctypes.data)
            if rc:
                break
            at += p.n_utts
        used = C.c_uint64()
        rc_end = L.ctts_gpu_session_end(h, C.byref(used))
        self._check(rc or rc_end)
        return off[:n], nbytes[:n], cnt[:n], int(used.value)

    def synth_pieces_g711(self, pieces: list[BatchPlan], params: AssemblyParams, law: int, out: np.ndarray):
        """A G.711 session of `law` (G711_ULAW or G711_ALAW) fed with the given plans, one piece each
        (ctts_gpu_session_begin_g711 / _submit_g711): one byte per sample in the uint8 buffer `out`, in the packed
        layout.  Returns (byte offsets, sample counts, bytes used) over all utterances of all pieces, in order."""
        assert out.dtype == np.uint8 and out.flags["C_CONTIGUOUS"]
        L = lib()
        h = C.c_void_p()
        self._check(L.ctts_gpu_session_begin_g711(self._h, C.byref(params), law, out.ctypes.data, out.size, None, None, C.byref(h)))
        n = sum(p.n_utts for p in pieces)
        off = np.zeros(max(n, 1), dtype=np.uint64)
        cnt = np.zeros(max(n, 1), dtype=np.uint32)
        at, rc = 0, 0
        for p in pieces:
            cp = p.as_c()
            rc = L.ctts_gpu_session_submit_g711(h, C.byref(cp), off[at:].ctypes.data, cnt[at:].ctypes.data)
            if rc:
                break
            at += p.n_utts
        used = C.c_uint64()
        rc_end = L.ctts_gpu_session_end(h, C.byref(used))
        self._check(rc or rc_end)
        return off[:n], cnt[:n], int(used.value)

    def flac_bound(self, plan: BatchPlan) -> int:
        """Bytes that are always enough for a FLAC session over the plan: ctts_gpu_flac_bound of every bound, rounded up to 16."""
        return sum((int(lib().ctts_gpu_flac_bound(int(b))) + 15) // 16 * 16 for b in self.bounds(plan))

    def synth_list(self, plan: BatchPlan, params: AssemblyParams) -> list[np.ndarray]:
        pcm, off, cnt = self.synth_batch(plan, params)
        return [pcm[int(off[u]):int(off[u]) + int(cnt[u])].copy() for u in range(plan.n_utts)]

    def create_plan(self, plan: BatchPlan, params: AssemblyParams, out_offsets: np.ndarray | None = None) -> ResidentPlan:
        h = C.c_void_p()
        cp = plan.as_c()
        off_ptr = None
        if out_offsets is not None:
            out_offsets = np.ascontiguousarray(out_offsets, dtype=np.uint64)
            off_ptr = out_offsets.ctypes.data
        self._check(lib().ctts_gpu_plan_create(self._h, C.byref(cp), C.byref(params), off_ptr, C.byref(h)))
        rp = ResidentPlan(self, h, plan.n_utts)
        self._plans.add(rp)
        return rp


def multi_synth_batch(ctxs: list[GpuSynth], plan: BatchPlan, params: AssemblyParams, pcm_out: np.ndarray | None = None,
                      out_offsets: np.ndarray | None = None):
    """ctts_gpu_multi_synth_batch: one batch partitioned over several contexts (one per GPU), every shard
    delivered into the caller's buffer at the utterance's own slot.  Returns (pcm, offsets, counts, shard_of)."""
    if out_offsets is None:
        out_offsets = ctxs[0].layout(plan)
    out_offsets = np.ascontiguousarray(out_offsets, dtype=np.uint64)
    total = int(out_offsets[-1])
    if pcm_out is None:
        pcm_out = np.empty(max(total, 1), dtype=np.int16)
    assert pcm_out.dtype == np.int16 and pcm_out.size >= total and pcm_out.flags["C_CONTIGUOUS"]
    counts = np.zeros(max(plan.n_utts, 1), dtype=np.uint32)
    shard_of = np.zeros(max(plan.n_utts, 1), dtype=np.uint32)
    arr = (C.c_void_p * len(ctxs))(*[c._h for c in ctxs])
    cp = plan.as_c()
    ctxs[0]._check(lib().ctts_gpu_multi_synth_batch(arr, len(ctxs), C.byref(cp), C.byref(params), pcm_out.ctypes.data,
                                                     out_offsets.ctypes.data, counts.ctypes.data, shard_of.ctypes.data))
    return pcm_out, out_offsets, counts[:plan.n_utts], shard_of[:plan.n_utts]
