"""GPU tests of the G.711 output (ctts_gpu_session_*_g711, ctts_b200_synth_texts_g711, the command line's g711=,
DESIGN.md 3.7): every utterance's bytes equal the oracle encoder (tests/g711_oracle.py) applied to the PCM a PCM session
delivers for the same pieces on the same context settings -- which the parity suites pin to the oracle -- in the packed
layout, with the law's silence code in the padding.

Run on a B200 with:  python -m pytest tests/test_gpu_g711.py -m gpu
"""
import ctypes as C
import shutil
import subprocess

import numpy as np
import pytest

import edge_voices as E
import g711_oracle as G

pytestmark = pytest.mark.gpu

ERR_INVALID_ARG, ERR_BOUNDS = -1, -101
LAWS = (G.ULAW, G.ALAW)
TABLE = {law: G.table(law) for law in LAWS}   # pinned to the reference by test_g711.py


def _enc(x, law):
    return TABLE[law][np.asarray(x, np.int16).astype(np.int64) + 32768]


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.fixture(scope="module")
def pipe(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.pipeline")


@pytest.fixture(scope="module")
def batch64(H, front_small):
    texts = H.corpus.batch(61, seed=4242, target_chars=90) + ["", "olá mundo", "São 1234 casas, não é?"]
    mixed = list(H.corpus.mixed_speeds(64, seed=17))
    mixed[::3] = [1.0] * len(mixed[::3])
    return texts, {"speed1": front_small.plan(texts), "mixed": front_small.plan(texts, mixed)}


def _capacity(g, pieces):
    return sum(int(((g.bounds(p).astype(np.int64) + 7) // 8 * 8).sum()) for p in pieces)


def _pcm_session(g, pieces, prm):
    buf = np.zeros(_capacity(g, pieces) + 8, np.int16)
    off, cnt = g.synth_pieces(pieces, prm, buf)
    return [buf[int(off[u]):int(off[u]) + int(cnt[u])].copy() for u in range(len(off))]


def _g711_session(g, pieces, prm, law, cap=None):
    out = np.full(max(_capacity(g, pieces) if cap is None else cap, 1), 0xA5, np.uint8)
    off, cnt, used = g.synth_pieces_g711(pieces, prm, law, out)
    return out, off, cnt, used


def _check(out, off, cnt, used, pcm, law, what):
    """The up8 layout, the counts, bytes_used, the codes and the silence padding of every utterance."""
    n = len(pcm)
    assert len(off) == n == len(cnt), what
    lengths = np.array([len(x) for x in pcm], np.int64)
    assert np.array_equal(cnt.astype(np.int64), lengths), f"{what}: counts"
    want_off = np.concatenate([[0], np.cumsum((lengths + 7) // 8 * 8)])
    assert np.array_equal(off.astype(np.int64), want_off[:-1]), f"{what}: offsets"
    assert used == int(want_off[-1]), f"{what}: bytes used"
    want = G.packed(pcm, law)
    got = out[:used].tobytes()
    if got != want:
        d = int(np.nonzero(np.frombuffer(got, np.uint8) != np.frombuffer(want, np.uint8))[0][0])
        u = int(np.searchsorted(want_off, d, side="right") - 1)
        raise AssertionError(f"{what}: first difference at byte {d}, utterance {u} ({len(pcm[u])} samples)")


@pytest.mark.parametrize("law", LAWS)
@pytest.mark.parametrize("hz", (8000, 11025, 16000, 22050))
@pytest.mark.parametrize("speeds", ("speed1", "mixed"))
def test_sessions_match_the_oracle(gpu, small_db, front_small, batch64, speeds, hz, law):
    plan = batch64[1][speeds]
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        g.set_output_rate(hz)
        for cuts in ([0, 64], [0, 1, 9, 9, 30, 31, 50, 64], list(range(0, 65, 4))):   # one piece, small pieces, > 4 pieces
            pieces = [plan.select(range(a, b)) for a, b in zip(cuts[:-1], cuts[1:])]
            pcm = _pcm_session(g, pieces, prm)
            assert any(len(x) % 8 for x in pcm)   # padding to write
            assert speeds != "speed1" or len(pcm[61]) == 0   # the empty text: a 0-sample utterance
            _check(*_g711_session(g, pieces, prm, law), pcm, law, f"{speeds} {hz} Hz law {law} cuts {len(cuts) - 1}")
    finally:
        g.close()


@pytest.mark.parametrize("law", LAWS)
@pytest.mark.parametrize("hz", (8000, 22050))
def test_loudness_settings(gpu, small_db, front_small, batch64, hz, law):
    plan = batch64[1]["mixed"]
    prm = front_small.params()
    pieces = [plan.select(range(0, 20)), plan.select(range(20, 64))]
    g = gpu.GpuSynth(small_db, 0)
    try:
        g.set_output_rate(hz)
        plain = _pcm_session(g, pieces, prm)
        for setting in ((-16.0, -1.0, False), (-23.0, -1.0, True), (0.0, -1.0, False)):
            g.set_loudness(*setting)
            pcm = _pcm_session(g, pieces, prm)
            if setting[0]:
                assert any(not np.array_equal(a, b) for a, b in zip(pcm, plain)), setting   # the stage did run
            _check(*_g711_session(g, pieces, prm, law), pcm, law, f"{hz} Hz loudness {setting}")
    finally:
        g.close()


@pytest.mark.parametrize("name", sorted(E.FAMILIES))
def test_edge_voices(gpu, name):
    fam = E.family(name)
    plan, prm = fam.plan(), fam.prm()
    g = gpu.GpuSynth(fam.db, 0)
    try:
        pcm = _pcm_session(g, [plan], prm)
        for u, x in enumerate(fam.expected()):
            assert np.array_equal(pcm[u], x), f"{name}: PCM of utterance {u}"
        for law in LAWS:
            _check(*_g711_session(g, [plan], prm, law), pcm, law, f"{name} law {law}")
    finally:
        g.close()


def test_full_scale_signals(gpu):
    """Signals delivered unchanged (noise over the whole int16 range, full-scale alternation, a ramp, tones) through
    both laws: both clipping ends and every segment of either sign (the code's top nibble) reach the encoder."""
    fam = E.signal_family("flac")
    plan, prm = fam.plan(), fam.prm()
    g = gpu.GpuSynth(fam.db, 0)
    try:
        pcm = _pcm_session(g, [plan], prm)
        x = np.concatenate(pcm).astype(np.int64)
        assert x.min() == -32768 and x.max() == 32767
        for law in LAWS:
            assert len(np.unique(_enc(x, law) >> 4)) == 16
            _check(*_g711_session(g, [plan], prm, law), pcm, law, f"full-scale signals law {law}")
    finally:
        g.close()


def test_piece_past_the_grid_limit(gpu):
    """One piece of 2 000 utterances and one of 70 000 (the encode grid splits at 65 535 utterances): the whole
    buffer equals the oracle, offsets and bytes used equal the up8 layout."""
    fam = E.signal_family("pieces")
    plan, prm = fam.plan(), fam.prm()
    sig = E.piece_signals()
    a, n = E.PIECE_SIZES[0], plan.n_utts
    assert n - a > 65535 and len(sig[0]) == 0
    g = gpu.GpuSynth(fam.db, 0)
    try:
        for law in LAWS:
            out, off, cnt, used = _g711_session(g, [plan.select(range(0, a)), plan.select(range(a, n))], prm, law)
            lengths = np.array([len(x) for x in sig], np.int64)[np.arange(n) % len(sig)]
            assert np.array_equal(cnt.astype(np.int64), lengths)
            ends = np.cumsum((lengths + 7) // 8 * 8)
            assert off[0] == 0 and np.array_equal(off[1:].astype(np.int64), ends[:-1]) and used == int(ends[-1])
            block = [np.concatenate([_enc(x, law), np.full((-len(x)) % 8, G.SILENCE[law], np.uint8)]) for x in sig]
            want = np.concatenate([block[u % len(sig)] for u in range(n)])
            assert np.array_equal(out[:used], want), f"law {law}"
    finally:
        g.close()


def test_too_small_capacity(gpu, small_db, front_small, batch64):
    plan = batch64[1]["speed1"]
    prm = front_small.params()
    pieces = [plan.select(range(a, a + 8)) for a in range(0, 64, 8)]
    g = gpu.GpuSynth(small_db, 0)
    try:
        for law in LAWS:
            pcm = _pcm_session(g, pieces, prm)
            _, _, _, used = _g711_session(g, pieces, prm, law)
            with pytest.raises(gpu.GpuError) as e:
                _g711_session(g, pieces, prm, law, cap=used - 1)
            assert f"error {ERR_BOUNDS}:" in str(e.value)
            # the context is usable afterwards, and the exact size is enough
            _check(*_g711_session(g, pieces, prm, law, cap=used), pcm, law, f"exact capacity law {law}")
    finally:
        g.close()


def test_invalid_calls(gpu, small_db, front_small, batch64):
    plan = batch64[1]["speed1"]
    prm = front_small.params()
    L = gpu.lib()
    g = gpu.GpuSynth(small_db, 0)
    try:
        cp = plan.as_c()
        o = np.zeros(64, np.uint64)
        b = np.zeros(64, np.uint32)
        c = np.zeros(64, np.uint32)
        pcm = np.zeros(_capacity(g, [plan]), np.int16)
        out = np.zeros(max(g.flac_bound(plan), pcm.size), np.uint8)
        h, h2 = C.c_void_p(), C.c_void_p()
        for law in (0, 3, -1, 7):
            assert L.ctts_gpu_session_begin_g711(g._h, C.byref(prm), law, out.ctypes.data, out.size, None, None, C.byref(h)) == ERR_INVALID_ARG
        # a PCM and a FLAC session take no G.711 submit, and no second session opens beside them
        for begin in (lambda: L.ctts_gpu_session_begin(g._h, C.byref(prm), pcm.ctypes.data, pcm.size, None, None, C.byref(h)),
                      lambda: L.ctts_gpu_session_begin_flac(g._h, C.byref(prm), out.ctypes.data, out.size, None, None, C.byref(h))):
            assert begin() == 0
            assert L.ctts_gpu_session_submit_g711(h, C.byref(cp), o.ctypes.data, c.ctypes.data) == ERR_INVALID_ARG
            assert L.ctts_gpu_session_begin_g711(g._h, C.byref(prm), G.ULAW, out.ctypes.data, out.size, None, None, C.byref(h2)) == ERR_INVALID_ARG
            assert L.ctts_gpu_session_end(h, None) == 0
        # a G.711 session takes no PCM or FLAC submit, and no second session of any kind
        for law in LAWS:
            assert L.ctts_gpu_session_begin_g711(g._h, C.byref(prm), law, out.ctypes.data, out.size, None, None, C.byref(h)) == 0
            assert L.ctts_gpu_session_submit(h, C.byref(cp), o.ctypes.data, c.ctypes.data) == ERR_INVALID_ARG
            assert L.ctts_gpu_session_submit_flac(h, C.byref(cp), o.ctypes.data, b.ctypes.data, c.ctypes.data) == ERR_INVALID_ARG
            assert L.ctts_gpu_session_begin_g711(g._h, C.byref(prm), law, out.ctypes.data, out.size, None, None, C.byref(h2)) == ERR_INVALID_ARG
            assert L.ctts_gpu_session_begin(g._h, C.byref(prm), pcm.ctypes.data, pcm.size, None, None, C.byref(h2)) == ERR_INVALID_ARG
            assert L.ctts_gpu_session_submit_g711(h, C.byref(cp), o.ctypes.data, c.ctypes.data) == 0
            used = C.c_uint64()
            assert L.ctts_gpu_session_end(h, C.byref(used)) == 0
            assert used.value == int(o[63]) + (int(c[63]) + 7) // 8 * 8
        # the context still delivers the same bytes
        want = _pcm_session(g, [plan], prm)
        for law in LAWS:
            _check(*_g711_session(g, [plan], prm, law), want, law, f"after the invalid calls, law {law}")
    finally:
        g.close()


def test_text_path_matches_the_session(gpu, pipe, small_db, front_small, batch64):
    texts, plans = batch64
    plan = plans["mixed"]
    speeds = np.asarray(plan.speed, np.float32)
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        for hz in (8000, 22050):
            g.set_output_rate(hz)
            batch = pipe.TextBatch(texts, speeds)
            cap = pipe.capacity_hint(front_small, batch, hz)
            pbuf = np.zeros(cap, np.int16)
            poff, pcnt, pused, _ = pipe.synth_texts(front_small, g, batch, pbuf)
            pcm = [pbuf[int(poff[u]):int(poff[u]) + int(pcnt[u])] for u in range(plan.n_utts)]
            assert all(np.array_equal(a, b) for a, b in zip(pcm, _pcm_session(g, [plan], prm)))
            for law in LAWS:
                for piece_utts, threads in ((16, 1), (192, 3)):
                    buf = np.full(cap, 0xA5, np.uint8)   # exactly ctts_b200_capacity_hint_rate bytes
                    off, cnt, used, tm = pipe.synth_texts_g711(front_small, g, batch, law, buf, piece_utts=piece_utts, threads=threads)
                    assert used == pused and tm.pieces >= 1
                    _check(buf, off, cnt, used, pcm, law, f"text path {hz} Hz law {law} pieces of {piece_utts}")
        with pytest.raises(gpu.GpuError):
            pipe.synth_texts_g711(front_small, g, pipe.TextBatch(texts[:2]), 3, np.zeros(1 << 20, np.uint8))
    finally:
        g.close()


def test_g711_header_symbols_are_exported(H, pipe):
    import os
    import test_abi
    names = test_abi._declared(os.path.join(H.ROOT, "include", "ctts_b200_g711.h"))
    assert names == ["ctts_b200_synth_texts_g711"]
    assert hasattr(pipe.lib(), names[0])
    names = test_abi._declared(os.path.join(H.ROOT, "include", "ctts_gpu.h"))
    for n in ("ctts_gpu_session_begin_g711", "ctts_gpu_session_submit_g711"):
        assert n in names and hasattr(H.importlib.import_module("2026-simple-c-tts_b200.gpu").lib(), n)


def test_command_line_writes_g711(H, small_db, tmp_path):
    b = H.importlib.import_module("2026-simple-c-tts_b200._build")
    exe = b.build_cli()
    shutil.copy(H.SHIPPED_YAML, tmp_path / "config.yaml")
    shutil.copy(H.NORM_CSV, tmp_path / "normalization.csv")
    (tmp_path / "voice.db").write_bytes(small_db)
    run = lambda *args: subprocess.run([exe, *args], cwd=tmp_path, capture_output=True, text=True)
    text = "olá mundo, bom dia"
    for extra in ([], ["1.5", "8000"], ["1.0", "16000", "lufs=-16"]):
        r = run("synth", "voice.db", text, "p.wav", *extra)
        assert r.returncode == 0, r.stderr
        wav = (tmp_path / "p.wav").read_bytes()
        pcm = np.frombuffer(wav[44:], "<i2")
        rate = int.from_bytes(wav[24:28], "little")
        for law, name in ((G.ULAW, "ulaw"), (G.ALAW, "alaw")):
            r = run("synth", "voice.db", text, f"{name}.wav", *extra, f"g711={name}")
            assert r.returncode == 0, r.stderr
            info = G.parse_wav((tmp_path / f"{name}.wav").read_bytes())
            assert info["law"] == law and info["rate"] == rate and info["count"] == len(pcm)
            assert np.array_equal(info["codes"], _enc(pcm, law)), (extra, name)
    (tmp_path / "t.tsv").write_text("1.0\tolá mundo\n1.5\tolá mundo\n1.0\t...\n0.7\tSão 1234 casas, não é?\n", encoding="utf-8")
    for args in (["w", "8000"], ["a", "8000", "g711=alaw"], ["u", "8000", "lufs=-20", "g711=ulaw", "dbtp=-2"], ["w2", "8000", "lufs=-20", "dbtp=-2"]):
        r = run("synth-batch", "voice.db", "t.tsv", *args)
        assert r.returncode == 0, r.stderr
    for u in range(4):
        for d, ref, law in (("a", "w", G.ALAW), ("u", "w2", G.ULAW)):
            pcm = np.frombuffer((tmp_path / ref / f"{u:06d}.wav").read_bytes()[44:], "<i2")
            info = G.parse_wav((tmp_path / d / f"{u:06d}.wav").read_bytes())
            assert info["law"] == law and info["rate"] == 8000 and np.array_equal(info["codes"], _enc(pcm, law)), (d, u)
    # usage errors: with FLAC, an unknown law, a repeated option
    for args in (["synth", "voice.db", text, "x.flac", "g711=ulaw"], ["synth", "voice.db", text, "x.wav", "g711=pcm"],
                 ["synth", "voice.db", text, "x.wav", "g711=ulaw", "g711=alaw"],
                 ["synth-batch", "voice.db", "t.tsv", "f", "8000", "flac", "g711=alaw"]):
        r = run(*args)
        assert r.returncode != 0 and "Usage" in r.stderr, args
