"""Test-side bindings: the CPU oracle (oracle/libctts_oracle.so), the compiled
reference (oracle/_ref/libctts_ref.so, built from /root/reference when present)
and shared fixtures.  Only tests/, smoke() and bench.py's baseline legs import this.
"""
from __future__ import annotations

import ctypes as C
import importlib
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

pkg = importlib.import_module("2026-simple-c-tts_b200")
front = importlib.import_module("2026-simple-c-tts_b200.front")
voicedb = importlib.import_module("2026-simple-c-tts_b200.voicedb")
corpus = importlib.import_module("2026-simple-c-tts_b200.corpus")

GOLDEN = os.path.join(ROOT, "tests", "golden")
SHIPPED_YAML = os.path.join(GOLDEN, "ctts_shipped.yaml")
NORM_CSV = os.path.join(GOLDEN, "normalization_rules.csv")
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "libctts_oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libctts_ref.so")
REF_BENCH = os.path.join(ORACLE_DIR, "_ref", "ctts_ref_bench")
REF_CLI = os.path.join(ORACLE_DIR, "_ref", "ctts")

MAX_UB_SPANS = 8


class OracleStats(C.Structure):
    _fields_ = [
        ("pre_count", C.c_uint64), ("out_count", C.c_uint64), ("trimmed", C.c_uint64),
        ("units", C.c_uint32), ("joins", C.c_uint32), ("pitch_shifts", C.c_uint32),
        ("contour_calls", C.c_uint32), ("wsola_frames", C.c_uint32), ("ub_spans", C.c_uint32),
        ("ub_span", (C.c_uint64 * 2) * MAX_UB_SPANS),
    ]


def build_oracle() -> None:
    subprocess.run(["make", "-C", ORACLE_DIR, "all"], check=True, stdout=subprocess.DEVNULL)


_oracle_lib = None


def oracle_lib() -> C.CDLL:
    global _oracle_lib
    if _oracle_lib is None:
        src = os.path.join(ORACLE_DIR, "ctts_oracle.c")
        if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src):
            subprocess.run(["make", "-C", ORACLE_DIR, "oracle"], check=True, stdout=subprocess.DEVNULL)
        L = C.CDLL(ORACLE_SO)
        i16p = C.POINTER(C.c_int16)
        L.ctts_oracle_open.argtypes = [C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t]
        L.ctts_oracle_close.argtypes = [C.c_void_p]
        L.ctts_oracle_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ctts_oracle_synth.argtypes = [C.c_void_p, C.POINTER(front.AssemblyParams), C.c_void_p, C.c_uint32,
                                        C.c_float, C.POINTER(i16p), C.POINTER(C.c_size_t),
                                        C.POINTER(i16p), C.POINTER(C.c_size_t), C.POINTER(OracleStats)]
        L.ctts_oracle_free.argtypes = [C.c_void_p]
        L.ctts_oracle_rms.argtypes = [C.c_void_p, C.c_size_t]
        L.ctts_oracle_rms.restype = C.c_float
        L.ctts_oracle_normalize_rms.argtypes = [C.c_void_p, C.c_size_t, C.c_float]
        L.ctts_oracle_remove_dc.argtypes = [C.c_void_p, C.c_size_t]
        L.ctts_oracle_estimate_pitch.argtypes = [C.c_void_p, C.c_size_t]
        L.ctts_oracle_estimate_pitch.restype = C.c_float
        L.ctts_oracle_smooth_pitch.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ctts_oracle_match_energy.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ctts_oracle_trim.argtypes = [C.c_void_p, C.c_size_t, C.c_float, C.c_size_t]
        L.ctts_oracle_trim.restype = C.c_size_t
        L.ctts_oracle_contour.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float,
                                          C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.ctts_oracle_contour.restype = C.c_uint32
        L.ctts_oracle_fade_in.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ctts_oracle_fade_out.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ctts_oracle_append.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                         C.c_size_t, C.c_size_t, C.c_int, C.c_int]
        L.ctts_oracle_append.restype = C.c_size_t
        L.ctts_oracle_wsola_offset.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        L.ctts_oracle_time_stretch.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_float,
                                               C.POINTER(i16p), C.POINTER(C.c_size_t), C.POINTER(C.c_uint32)]
        _oracle_lib = L
    return _oracle_lib


class Oracle:
    """CPU restatement of the assembly hot path (oracle/ctts_oracle.c)."""

    def __init__(self, voice_db: bytes):
        self._buf = (C.c_char * len(voice_db)).from_buffer_copy(voice_db)
        h = C.c_void_p()
        rc = oracle_lib().ctts_oracle_open(C.byref(h), C.addressof(self._buf), len(voice_db))
        if rc:
            raise RuntimeError(f"ctts_oracle_open: {rc}")
        self._h = h

    def __del__(self):
        try:
            if self._h:
                oracle_lib().ctts_oracle_close(self._h)
                self._h = None
        except Exception:
            pass

    def tables(self):
        luts = np.zeros(3 * 1024, np.float32)
        h256 = np.zeros(256, np.float32)
        h512 = np.zeros(512, np.float32)
        oracle_lib().ctts_oracle_tables(self._h, luts.ctypes.data, h256.ctypes.data, h512.ctypes.data)
        return luts, h256, h512

    def synth(self, params, ops: np.ndarray, speed: float = 1.0, want_pre: bool = False):
        """Returns (pcm, stats[, pre])."""
        L = oracle_lib()
        ops = np.ascontiguousarray(ops)
        out = C.POINTER(C.c_int16)()
        n = C.c_size_t()
        pre = C.POINTER(C.c_int16)()
        npre = C.c_size_t()
        st = OracleStats()
        rc = L.ctts_oracle_synth(self._h, C.byref(params), ops.ctypes.data, len(ops), C.c_float(speed),
                                 C.byref(out), C.byref(n), C.byref(pre) if want_pre else None,
                                 C.byref(npre) if want_pre else None, C.byref(st))
        if rc:
            raise RuntimeError(f"ctts_oracle_synth: {rc}")
        pcm = np.ctypeslib.as_array(out, shape=(max(n.value, 1),))[:n.value].copy()
        L.ctts_oracle_free(out)
        if want_pre:
            p = np.ctypeslib.as_array(pre, shape=(max(npre.value, 1),))[:npre.value].copy()
            L.ctts_oracle_free(pre)
            return pcm, st, p
        return pcm, st

    def synth_plan(self, params, plan, want_stats: bool = False):
        outs, stats = [], []
        for u in range(plan.n_utts):
            pcm, st = self.synth(params, plan.utt_ops(u), float(plan.speed[u]))
            outs.append(pcm)
            stats.append(st)
        return (outs, stats) if want_stats else outs


def ub_mask(st: OracleStats, n: int) -> np.ndarray:
    """Boolean mask of samples whose reference value depends on an out-of-bounds heap read."""
    m = np.zeros(n, dtype=bool)
    for k in range(min(int(st.ub_spans), MAX_UB_SPANS)):
        lo, hi = int(st.ub_span[k][0]), int(st.ub_span[k][1])
        m[lo:min(hi, n)] = True
    return m


# ------------------------------------------------------------------ reference

def have_reference() -> bool:
    return os.path.exists(REF_SO)


_ref_lib = None


def ref_lib() -> C.CDLL:
    global _ref_lib
    if _ref_lib is None:
        L = C.CDLL(REF_SO)
        i16p = C.POINTER(C.c_int16)
        L.ref_open.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
        L.ref_synth.argtypes = [C.c_char_p, C.c_float, C.POINTER(i16p), C.POINTER(C.c_size_t)]
        L.ref_free.argtypes = [C.c_void_p]
        L.ref_unit_trace.argtypes = [C.c_char_p]
        L.ref_unit_trace.restype = C.c_void_p
        L.ref_normalized_text.argtypes = [C.c_char_p]
        L.ref_normalized_text.restype = C.c_void_p
        L.ref_rule_count.restype = C.c_size_t
        L.ref_get_config.argtypes = [C.POINTER(front.Config)]
        L.ref_set_config.argtypes = [C.POINTER(front.Config)]
        L.ref_fade_luts.argtypes = [C.c_void_p]
        L.ref_hann256.argtypes = [C.c_void_p]
        L.ref_hann512.argtypes = [C.c_void_p]
        L.ref_normalize_rms.argtypes = [C.c_void_p, C.c_size_t, C.c_float]
        L.ref_calculate_rms.argtypes = [C.c_void_p, C.c_size_t]
        L.ref_calculate_rms.restype = C.c_float
        L.ref_remove_dc_offset.argtypes = [C.c_void_p, C.c_size_t]
        L.ref_estimate_pitch.argtypes = [C.c_void_p, C.c_size_t]
        L.ref_estimate_pitch.restype = C.c_float
        L.ref_smooth_pitch_boundary.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ref_match_boundary_energy.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t]
        L.ref_remove_silence_regions.argtypes = [C.c_void_p, C.c_size_t, C.c_float, C.c_size_t]
        L.ref_remove_silence_regions.restype = C.c_size_t
        L.ref_apply_smooth_pitch_contour.argtypes = [C.c_void_p, C.c_size_t, C.c_float, C.c_float]
        L.ref_apply_fade_in.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t]
        L.ref_apply_fade_out.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t]
        L.ref_apply_phrase_intonation.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_float]
        L.ref_append_crossfade.argtypes = [C.c_void_p, C.POINTER(C.c_size_t), C.c_size_t, C.c_void_p,
                                           C.c_size_t, C.c_float, C.c_int]
        L.ref_time_stretch.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(i16p), C.POINTER(C.c_size_t), C.c_float]
        L.ref_wsola_offset.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
        L.ref_cross_correlation.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.ref_cross_correlation.restype = C.c_float
        L.ref_build_database.argtypes = [C.c_char_p, C.c_char_p]
        _ref_lib = L
    return _ref_lib


class Reference:
    """The compiled, unmodified reference engine (one per process: it keeps global state)."""

    def __init__(self, db_path: str, config_path: str | None = SHIPPED_YAML, norm_csv: str | None = NORM_CSV):
        L = ref_lib()
        # the reference prints one warning per rule glibc rejects; keep test logs readable
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(2)
        os.dup2(devnull, 2)
        try:
            rc = L.ref_open(db_path.encode(), config_path.encode() if config_path else None,
                            norm_csv.encode() if norm_csv else None)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            os.close(devnull)
        if rc:
            raise RuntimeError("ref_open failed")

    def synth(self, text: str, speed: float = 1.0) -> np.ndarray:
        L = ref_lib()
        out = C.POINTER(C.c_int16)()
        n = C.c_size_t()
        rc = L.ref_synth(text.encode("utf-8"), C.c_float(speed), C.byref(out), C.byref(n))
        if rc:
            raise RuntimeError(f"ctts_synthesize: {rc}")
        pcm = np.ctypeslib.as_array(out, shape=(max(n.value, 1),))[:n.value].copy()
        L.ref_free(out)
        return pcm

    def unit_trace(self, text: str) -> list[str]:
        L = ref_lib()
        p = L.ref_unit_trace(text.encode("utf-8"))
        s = C.string_at(p).decode("utf-8", errors="replace")
        L.ref_free(p)
        return [t[1:-1] for t in s.split() if t.startswith("[") and t.endswith("]")]

    def normalized_text(self, text: str) -> str:
        L = ref_lib()
        p = L.ref_normalized_text(text.encode("utf-8"))
        s = C.string_at(p).decode("utf-8", errors="replace")
        L.ref_free(p)
        return s

    def config(self):
        c = front.Config()
        ref_lib().ref_get_config(C.byref(c))
        return c

    def set_config(self, c) -> None:
        ref_lib().ref_set_config(C.byref(c))


# ------------------------------------------------------------------- fixtures

_db_cache: dict = {}


def synthetic_db(n_syllables: int = 1749, seed: int = 2026) -> bytes:
    key = (n_syllables, seed)
    if key not in _db_cache:
        _db_cache[key] = voicedb.synthetic_voice_db(n_syllables, seed)
    return _db_cache[key]


def small_db() -> bytes:
    """A reduced voice (all open syllables, ~11 MB) that builds in about a second."""
    return synthetic_db(1100, 2026)


def shipped_config():
    return front.load_config(SHIPPED_YAML)


GOLDEN_VECTORS = os.path.join(GOLDEN, "ref_vectors.npz.xz")


def save_golden_vectors(arrays: dict) -> None:
    """Writes tests/golden/ref_vectors.npz.xz: an uncompressed .npz in one xz stream, every int16 array (all PCM)
    stored as its first differences along the last axis.  Both make the file about half the size of
    np.savez_compressed's."""
    import io
    import lzma
    buf = io.BytesIO()
    np.savez(buf, **{k: np.diff(v, prepend=np.int16(0)) if v.dtype == np.int16 else v for k, v in arrays.items()})
    with open(GOLDEN_VECTORS, "wb") as f:
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))


def golden_vectors() -> dict:
    """tests/golden/ref_vectors.npz.xz (make_golden.py), decoded: per-stage vectors and end-to-end PCM of the
    compiled reference."""
    import io
    import lzma
    with lzma.open(GOLDEN_VECTORS) as f:
        z = np.load(io.BytesIO(f.read()), allow_pickle=False)
        return {k: np.cumsum(v, axis=-1, dtype=np.int16) if v.dtype == np.int16 else v for k, v in z.items()}


def golden_corpus() -> dict:
    """tests/golden/ref_corpus.json: SHA-1 / length of the compiled reference's PCM (make_golden_corpus.py)."""
    import json
    with open(os.path.join(GOLDEN, "ref_corpus.json"), encoding="utf-8") as f:
        return json.load(f)


def masked_sha1(pcm: np.ndarray, mask: np.ndarray) -> str:
    import hashlib
    x = np.ascontiguousarray(pcm, dtype="<i2").copy()
    x[mask[:len(x)]] = 0
    return hashlib.sha1(x.tobytes()).hexdigest()


def odd_offset_voice() -> bytes:
    """The small voice plus one unit whose text makes the string pool's size odd, so that the PCM pool starts
    at an odd byte offset of voice.db (ctts.c:1001-1004, :1159).  Same construction as make_golden_corpus.py."""
    key = "odd"
    if key not in _db_cache:
        vdb = voicedb.parse_voice_db(small_db())
        units = [(vdb.unit_text(i), vdb.unit_pcm(i)) for i in range(vdb.unit_count)]
        rng = np.random.default_rng(4)
        for extra in ("zzq", "zzqq"):
            db = voicedb.build_voice_db(units + [(extra, (rng.normal(0, 2000, 3000)).astype(np.int16))])
            if voicedb.parse_voice_db(db).audio_offset % 2 == 1:
                _db_cache[key] = db
                break
        else:
            raise AssertionError("could not make the audio offset odd")
    return _db_cache[key]
