"""The CPU oracle (oracle/ctts_oracle.c) pinned to the reference: committed golden vectors made by the
compiled reference (tests/golden/make_golden.py) and, where oracle/_ref exists, the reference itself."""
import ctypes as C

import numpy as np
import pytest


def _i16(a):
    return np.ascontiguousarray(a, dtype=np.int16)


def test_golden_vector_encoding_round_trips(H, tmp_path, monkeypatch):
    """ref_vectors.npz.xz stores int16 arrays as first differences: they must decode exactly, whatever their shape."""
    monkeypatch.setattr(H, "GOLDEN_VECTORS", str(tmp_path / "v.npz.xz"))
    rng = np.random.default_rng(0)
    arrays = {"pcm": rng.integers(-32768, 32768, 1000).astype(np.int16), "empty": np.zeros(0, np.int16),
              "frames": rng.integers(-32768, 32768, (3, 50)).astype(np.int16), "f": rng.random(7).astype(np.float32)}
    H.save_golden_vectors(arrays)
    got = H.golden_vectors()
    assert set(got) == set(arrays)
    for k, v in arrays.items():
        assert got[k].dtype == v.dtype and got[k].shape == v.shape and np.array_equal(got[k], v), k


def test_tables_match_reference_bitwise(oracle_small, golden):
    luts, h256, h512 = oracle_small.tables()
    assert np.array_equal(luts.view(np.uint32), golden["luts"].view(np.uint32))
    assert np.array_equal(h256.view(np.uint32), golden["hann256"].view(np.uint32))
    assert np.array_equal(h512.view(np.uint32), golden["hann512"].view(np.uint32))


def test_unit_stages_match_golden(H, oracle_small, golden, small_db):
    L = H.oracle_lib()
    db = H.voicedb.parse_voice_db(small_db)
    units = [_i16(db.unit_pcm(int(i)).copy()) for i in golden["stage_units"]]
    norm = []
    for k, u in enumerate(units):
        assert np.float32(L.ctts_oracle_rms(u.ctypes.data, len(u))) == golden["rms"][k]
        x = u.copy()
        L.ctts_oracle_normalize_rms(x.ctypes.data, len(x), C.c_float(3000.0))
        assert np.array_equal(x, golden[f"normalize_{k}"])
        norm.append(x)
        y = x.copy()
        L.ctts_oracle_remove_dc(y.ctypes.data, len(y))
        assert np.array_equal(y, golden[f"dc_{k}"])
        assert np.float32(L.ctts_oracle_estimate_pitch(x.ctypes.data, min(len(x) // 2, 3968))) == golden["pitch_head"][k]
        t = _i16(x[len(x) - 1300:])
        assert np.float32(L.ctts_oracle_estimate_pitch(t.ctypes.data, 1300)) == golden["pitch_tail"][k]
    for k in range(len(units) - 1):
        for xf in (1984, 396):
            prev = _i16(golden[f"dc_{k}"])
            nxt = norm[k + 1].copy()
            L.ctts_oracle_smooth_pitch(prev.ctypes.data, len(prev), nxt.ctypes.data, len(nxt), xf)
            assert np.array_equal(nxt, golden[f"smooth_{k}_{xf}"])
            L.ctts_oracle_match_energy(prev.ctypes.data, len(prev), nxt.ctypes.data, len(nxt), xf)
            assert np.array_equal(nxt, golden[f"match_{k}_{xf}"])


def test_trim_contour_fades_match_golden(H, oracle_small, golden):
    L = H.oracle_lib()
    x = _i16(golden["trim_in"]).copy()
    n = L.ctts_oracle_trim(x.ctypes.data, len(x), C.c_float(0.04), 771)
    assert n == len(golden["trim_out"]) < len(x)
    assert np.array_equal(x[:n], golden["trim_out"])
    for k in range(3):
        f0, f1 = [float(v) for v in golden[f"contour_{k}_f"]]
        y = _i16(golden["trim_out"]).copy()
        lo, hi = C.c_size_t(), C.c_size_t()
        L.ctts_oracle_contour(oracle_small._h, y.ctypes.data, len(y), C.c_float(f0), C.c_float(f1), C.byref(lo), C.byref(hi))
        want = golden[f"contour_{k}"]
        mask = np.ones(len(y), bool)
        mask[lo.value:hi.value] = False          # samples the reference computed from out-of-bounds reads
        assert np.array_equal(y[mask], want[mask])
        assert hi.value - lo.value <= 32
    y = _i16(golden["dc_3"]).copy()
    L.ctts_oracle_fade_in(oracle_small._h, y.ctypes.data, len(y), 66)
    L.ctts_oracle_fade_out(oracle_small._h, y.ctypes.data, len(y), 66)
    assert np.array_equal(y, golden["fades"])


def test_phrase_intonation_matches_golden(H, oracle_small, golden, front_small):
    # drive the oracle's WORD_END executor with the front end's scalars for every phrase type / word position
    F = H.front
    prm = front_small.params()
    region = _i16(golden["trim_out"])
    for pt in range(4):
        for wi, tw in ((0, 5), (2, 5), (3, 5), (4, 5), (0, 1)):
            op = front_small.word_end_op(pt, wi, tw)[0]
            got = _apply_word_end(H, oracle_small, prm, region, op)
            want = golden[f"inton_{pt}_{wi}_{tw}"]
            diff = np.nonzero(got != want)[0]
            # differences may only sit where the reference read out of bounds (tail of a contour call)
            assert len(diff) <= 40, (pt, wi, tw, len(diff))


def _apply_word_end(H, oracle, prm, region, op):
    """Runs [raw region via a fake unit] is not possible; emulate with the stage API instead."""
    import ctypes as C
    L = H.oracle_lib()
    F = H.front
    x = region.copy()
    n = len(x)
    flags = int(op["flags"])
    if not (flags & F.WE_INTON) or n < 100:
        return x
    lo, hi = C.c_size_t(), C.c_size_t()
    done = False
    if flags & F.WE_CIRCUMFLEX:
        rise = int(np.float32(n) * np.float32(0.6))
        if rise > 100 and n - rise > 100:
            a = _i16(x[:rise]).copy()
            b = _i16(x[rise:]).copy()
            L.ctts_oracle_contour(oracle._h, a.ctypes.data, len(a), C.c_float(op["f0"]), C.c_float(op["f2"]), C.byref(lo), C.byref(hi))
            L.ctts_oracle_contour(oracle._h, b.ctypes.data, len(b), C.c_float(op["f2"]), C.c_float(op["f1"]), C.byref(lo), C.byref(hi))
            x = np.concatenate([a, b])
            done = True
    if not done:
        L.ctts_oracle_contour(oracle._h, x.ctypes.data, n, C.c_float(op["f0"]), C.c_float(op["f1"]), C.byref(lo), C.byref(hi))
    if flags & F.WE_ENERGY:
        i = np.arange(n, dtype=np.float32)
        t = i / np.float32(n - 1)
        e = np.float32(op["e0"]) + (np.float32(op["e1"]) - np.float32(op["e0"])) * t
        v = x.astype(np.float32) * e
        v = np.minimum(v, np.float32(32767.0))
        v = np.maximum(v, np.float32(-32768.0))
        x = v.astype(np.int32).astype(np.int16)
    return x


def test_wsola_matches_golden_and_known_lengths(H, oracle_small, golden):
    L = H.oracle_lib()
    sig = _i16(golden["wsola_in"])
    for sp in (0.5, 0.7, 1.5, 2.0):
        o = C.POINTER(C.c_int16)()
        n = C.c_size_t()
        fr = C.c_uint32()
        rc = L.ctts_oracle_time_stretch(oracle_small._h, sig.ctypes.data, len(sig), C.c_float(sp), C.byref(o), C.byref(n), C.byref(fr))
        assert rc == 0
        got = np.ctypeslib.as_array(o, shape=(max(n.value, 1),))[:n.value].copy()
        L.ctts_oracle_free(o)
        assert np.array_equal(got, golden[f"wsola_{sp}"])
    # known answers from the reference's shipped docs/audio/{100,104,102,97}_speed_*.wav (SURVEY.md section 4):
    # 73 930 samples in -> (574-1)*hop+512 out before the trailing-zero trim
    rng = np.random.default_rng(0)
    x = _i16(rng.integers(-3000, 3000, 73930))
    x[-600:] = np.where(x[-600:] == 0, 1, x[-600:])
    for sp, want in ((2.0, 37184), (1.5, 49217), (0.5, 147200)):
        o = C.POINTER(C.c_int16)()
        n = C.c_size_t()
        fr = C.c_uint32()
        L.ctts_oracle_time_stretch(oracle_small._h, x.ctypes.data, len(x), C.c_float(sp), C.byref(o), C.byref(n), C.byref(fr))
        L.ctts_oracle_free(o)
        assert fr.value == 574
        assert want - 64 <= n.value <= want   # only trailing zeros may be stripped


def test_end_to_end_matches_golden_pcm(H, oracle_small, front_small, golden):
    texts = [str(t) for t in golden["e2e_texts"]]
    speeds = [float(s) for s in golden["e2e_speeds"]]
    plan = front_small.plan(texts, speeds)
    prm = front_small.params()
    for k in range(len(texts)):
        got, st, pre = oracle_small.synth(prm, plan.utt_ops(k), speeds[k], want_pre=True)
        want = golden[f"e2e_pcm_{k}"]
        assert len(got) == len(want), (texts[k], len(got), len(want))
        if speeds[k] == 1.0:
            mask = ~H.ub_mask(st, len(got))
            assert np.array_equal(got[mask], want[mask]), texts[k]
        elif st.ub_spans == 0:
            assert np.array_equal(got, want), texts[k]
        else:
            assert np.mean(got != want) < 1e-3


def test_oracle_vs_live_reference(H, oracle_small, front_small, reference_small):
    texts = ["olá mundo", "a", " ", "", "..."] + H.corpus.batch(24, seed=77)
    prm = front_small.params()
    total = diff = 0
    for sp in (1.0, 1.3):
        plan = front_small.plan(texts, [sp] * len(texts))
        for k, t in enumerate(texts):
            want = reference_small.synth(t, sp)
            got, st = oracle_small.synth(prm, plan.utt_ops(k), sp)
            assert len(got) == len(want), (t, sp)
            total += len(got)
            if sp == 1.0:
                d = got != want
                assert not (d & ~H.ub_mask(st, len(got))).any(), t   # every mismatch is a reference out-of-bounds read
                diff += int(d.sum())
            elif st.ub_spans == 0:
                assert np.array_equal(got, want), (t, sp)
    assert diff / max(total, 1) < 1e-4


def test_oracle_matches_reference_hashes_of_corpus_sentences(H, small_db, front_small, oracle_small):
    """tests/golden/ref_corpus.json holds SHA-1 + length of the COMPILED REFERENCE's PCM for 48 sentences of the
    benchmark corpus (32 at speed 1.0, 16 stretched) -- made where the reference tree exists, checked here (and
    against the CUDA path in test_gpu_parity.py) where it does not."""
    import hashlib
    G = H.golden_corpus()
    assert G["voice_sha256"] == hashlib.sha256(small_db).hexdigest()
    rows = G["corpus"]
    assert len(rows) >= 48 and sum(r["speed"] != 1.0 for r in rows) >= 16
    prm = front_small.params()
    plan = front_small.plan([r["text"] for r in rows], [r["speed"] for r in rows])
    for u, r in enumerate(rows):
        got, st = oracle_small.synth(prm, plan.utt_ops(u), r["speed"])
        assert len(got) == r["samples"], r["text"]
        assert H.masked_sha1(got, H.ub_mask(st, len(got))) == r["sha1"], r["text"]


def test_oracle_on_a_voice_with_an_odd_pcm_offset(H):
    """voice.db whose PCM pool starts at an odd byte offset (the reference reads it through a misaligned
    int16_t*, ctts.c:1159): the oracle reproduces the compiled reference's hashes."""
    import hashlib
    db = H.odd_offset_voice()
    assert H.voicedb.parse_voice_db(db).audio_offset % 2 == 1
    G = H.golden_corpus()
    assert G["odd_voice_sha256"] == hashlib.sha256(db).hexdigest()
    fr = H.front.Front(db, H.shipped_config(), H.NORM_CSV)
    prm = fr.params()
    orc = H.Oracle(db)
    rows = G["odd_voice"]
    plan = fr.plan([r["text"] for r in rows], [r["speed"] for r in rows])
    for u, r in enumerate(rows):
        got, st = orc.synth(prm, plan.utt_ops(u), r["speed"])
        assert len(got) == r["samples"] and H.masked_sha1(got, H.ub_mask(st, len(got))) == r["sha1"], r["text"]
