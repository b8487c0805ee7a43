"""Generates tests/golden/ref_vectors.npz.xz from the COMPILED, UNMODIFIED reference
(oracle/_ref/libctts_ref.so, built from the reference's ctts.c by oracle/Makefile).

Run where the reference tree exists:   python tests/golden/make_golden.py
The fixture travels to the GPU box (the reference tree does not) and pins the
oracle and the CUDA path to outputs of the reference itself: end-to-end PCM for
a few utterances and per-stage vectors from the reference's static functions.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import harness as H  # noqa: E402

E2E = [
    ("olá mundo", 1.0),
    ("olá mundo", 1.5),
    ("Olá, mundo! Como vai você?", 1.0),
    ("O Brasil tem 27 estados e a música é boa.", 1.0),
    ("Dr. Rosa mora a 12 km da praia; a casa é azul, verde e branca!", 1.0),
    ("A ideia do rei era feia?", 0.7),
    ("rato rua rio", 2.0),
    ("xyz @ 7", 1.0),
    ("", 1.0),
    ("casa", 1.2),
]


def i16(a):
    return np.ascontiguousarray(a, dtype=np.int16)


def main() -> None:
    assert H.have_reference(), "build oracle/_ref first (make -C oracle ref)"
    L = H.ref_lib()
    db = H.small_db()
    out = {"db_sha256": np.frombuffer(hashlib.sha256(db).digest(), dtype=np.uint8)}
    with tempfile.TemporaryDirectory() as d:
        dbp = os.path.join(d, "voice.db")
        with open(dbp, "wb") as f:
            f.write(db)
        ref = H.Reference(dbp)
        out["e2e_texts"] = np.array([t for t, _ in E2E])
        out["e2e_speeds"] = np.array([s for _, s in E2E], dtype=np.float32)
        for k, (t, s) in enumerate(E2E):
            out[f"e2e_pcm_{k}"] = ref.synth(t, s)
            out[f"e2e_units_{k}"] = np.array(ref.unit_trace(t) or [""])
            out[f"e2e_norm_{k}"] = np.array(ref.normalized_text(t))
        out["rule_count"] = np.array([L.ref_rule_count()], dtype=np.int64)

        vdb = H.voicedb.parse_voice_db(db)
        pick = [3, 40, 200, 555, 800, 1000]
        units = [i16(vdb.unit_pcm(i).copy()) for i in pick]
        out["stage_units"] = np.array(pick, dtype=np.int64)

        # tables
        luts = np.zeros(3 * 1024, np.float32)
        h256 = np.zeros(256, np.float32)
        h512 = np.zeros(512, np.float32)
        L.ref_fade_luts(luts.ctypes.data)
        L.ref_hann256(h256.ctypes.data)
        L.ref_hann512(h512.ctypes.data)
        out["luts"], out["hann256"], out["hann512"] = luts, h256, h512

        norm = []
        for k, u in enumerate(units):
            x = u.copy()
            L.ref_normalize_rms(x.ctypes.data, len(x), C.c_float(3000.0))
            norm.append(x)
            out[f"normalize_{k}"] = x
            y = x.copy()
            L.ref_remove_dc_offset(y.ctypes.data, len(y))
            out[f"dc_{k}"] = y
        out["rms"] = np.array([L.ref_calculate_rms(u.ctypes.data, len(u)) for u in units], dtype=np.float32)
        out["pitch_head"] = np.array([L.ref_estimate_pitch(x.ctypes.data, min(len(x) // 2, 3968)) for x in norm],
                                     dtype=np.float32)
        out["pitch_tail"] = np.array(
            [L.ref_estimate_pitch(x[len(x) - 1300:].ctypes.data, 1300) for x in norm], dtype=np.float32)

        # joins: prev = dc-removed normalised unit, next = normalised unit
        for k in range(len(units) - 1):
            for xf in (1984, 396):
                prev = out[f"dc_{k}"].copy()
                nxt = norm[k + 1].copy()
                L.ref_smooth_pitch_boundary(prev.ctypes.data, len(prev), nxt.ctypes.data, len(nxt), xf)
                out[f"smooth_{k}_{xf}"] = nxt.copy()
                L.ref_match_boundary_energy(prev.ctypes.data, len(prev), nxt.ctypes.data, len(nxt), xf)
                out[f"match_{k}_{xf}"] = nxt.copy()

        # a word region: three units, a comma pause in the middle (long silent run), DC removed
        region = np.concatenate([out["dc_0"], np.zeros(2381, np.int16), out["dc_1"], out["dc_2"]])
        x = region.copy()
        n_new = L.ref_remove_silence_regions(x.ctypes.data, len(x), C.c_float(0.04), 771)
        out["trim_in"] = region
        out["trim_out"] = x[:n_new].copy()
        for k, (f0, f1) in enumerate([(0.9702, 1.0098), (1.1, 1.0444), (1.02, 0.94)]):
            y = out["trim_out"].copy()
            L.ref_apply_smooth_pitch_contour(y.ctypes.data, len(y), C.c_float(f0), C.c_float(f1))
            out[f"contour_{k}"] = y
            out[f"contour_{k}_f"] = np.array([f0, f1], dtype=np.float32)
        for pt in range(4):
            for wi, tw in ((0, 5), (2, 5), (3, 5), (4, 5), (0, 1)):
                y = out["trim_out"].copy()
                L.ref_apply_phrase_intonation(y.ctypes.data, len(y), pt, wi, tw, C.c_float(0.10))
                out[f"inton_{pt}_{wi}_{tw}"] = y
        y = out["dc_3"].copy()
        L.ref_apply_fade_in(y.ctypes.data, len(y), 66)
        L.ref_apply_fade_out(y.ctypes.data, len(y), 66)
        out["fades"] = y

        # WSOLA
        sig = np.concatenate([out["dc_0"], out["dc_1"], np.zeros(1323, np.int16), out["dc_2"], out["dc_4"]])
        out["wsola_in"] = sig
        for sp in (0.5, 0.7, 1.5, 2.0):
            o = C.POINTER(C.c_int16)()
            n = C.c_size_t()
            rc = L.ref_time_stretch(sig.ctypes.data, len(sig), C.byref(o), C.byref(n), C.c_float(sp))
            assert rc == 0
            out[f"wsola_{sp}"] = np.ctypeslib.as_array(o, shape=(max(n.value, 1),))[:n.value].copy()
            L.ref_free(o)
    H.save_golden_vectors(out)
    print("wrote", H.GOLDEN_VECTORS, os.path.getsize(H.GOLDEN_VECTORS), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
