"""GPU tests of the FLAC output (ctts_gpu_session_*_flac, ctts_b200_synth_texts_flac, DESIGN.md 3.5): every file the
device writes is byte-identical to the oracle encoder (tests/flac_oracle.c) applied to the PCM a PCM session delivers
for the same plan -- which the parity suite pins to the oracle -- and decodes through the independent decoder
(tests/flac_decode.c) to that PCM.

Run on a B200 with:  python -m pytest tests/test_gpu_flac.py -m gpu
"""
import ctypes as C
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import edge_voices as E
import flac_codec as F

pytestmark = pytest.mark.gpu

ERR_INVALID_ARG, ERR_BOUNDS = -1, -101
ODD_RATE = 11025   # no RFC rate code: 16-bit Hz in every frame header


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.fixture(scope="module")
def pipe(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.pipeline")


def _pcm_session(g, pieces, prm):
    n = sum(p.n_utts for p in pieces)
    cap = sum(int(((g.bounds(p).astype(np.int64) + 7) // 8 * 8).sum()) for p in pieces) + 8
    buf = np.zeros(cap, np.int16)
    off, cnt = g.synth_pieces(pieces, prm, buf)
    assert len(off) == n
    return [buf[int(off[u]):int(off[u]) + int(cnt[u])].copy() for u in range(n)]


def _flac_session(g, pieces, prm, cap=None):
    if cap is None:
        cap = sum(g.flac_bound(p) for p in pieces)
    out = np.full(max(cap, 1), 0xA5, np.uint8)
    off, nbytes, cnt, used = g.synth_pieces_flac(pieces, prm, out)
    return out, off, nbytes, cnt, used


def _check_files(out, off, nbytes, cnt, used, pcm, hz, what, decode=True):
    """Layout, oracle bytes and decoded samples of every file."""
    n = len(pcm)
    assert len(off) == n == len(nbytes) == len(cnt)
    at = 0
    for u in range(n):
        assert int(off[u]) == at, f"{what}: utterance {u} at {int(off[u])}, expected {at}"
        assert int(cnt[u]) == len(pcm[u]), f"{what}: utterance {u} count"
        end = at + int(nbytes[u])
        pad = (end + 15) // 16 * 16
        assert not out[end:pad].any(), f"{what}: padding of utterance {u} is not zero"
        at = pad
    assert used == at
    files = [out[int(off[u]):int(off[u]) + int(nbytes[u])].tobytes() for u in range(n)]
    with ThreadPoolExecutor(max(1, min(32, os.cpu_count() or 1))) as ex:
        want = list(ex.map(lambda x: F.encode(x, hz), pcm))
    for u in range(n):
        if files[u] != want[u]:
            a, b = np.frombuffer(files[u], np.uint8), np.frombuffer(want[u], np.uint8)
            k = min(len(a), len(b))
            d = np.nonzero(a[:k] != b[:k])[0]
            raise AssertionError(f"{what}: file of utterance {u} ({len(pcm[u])} samples) differs from the oracle: "
                                 f"{len(a)} vs {len(b)} bytes, first difference at byte {d[0] if len(d) else k}")
        if decode:
            got, info = F.decode(files[u])
            assert np.array_equal(got, pcm[u]) and info["sample_rate"] == hz, f"{what}: decoding utterance {u}"
    return files


@pytest.fixture(scope="module")
def batch64(H, front_small):
    texts = H.corpus.batch(61, seed=4242, target_chars=90) + ["", "olá mundo", "São 1234 casas, não é?"]
    mixed = list(H.corpus.mixed_speeds(64, seed=17))
    mixed[::3] = [1.0] * len(mixed[::3])
    return texts, {"speed1": front_small.plan(texts), "mixed": front_small.plan(texts, mixed)}


@pytest.mark.parametrize("speeds", ("speed1", "mixed"))
def test_batch64_matches_the_oracle(gpu, small_db, front_small, batch64, speeds):
    plan = batch64[1][speeds]
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        for cuts in ([0, 64], [0, 1, 9, 9, 30, 31, 50, 64], list(range(0, 65, 4))):   # one piece, small pieces, > 4 pieces
            pieces = [plan.select(range(a, b)) for a, b in zip(cuts[:-1], cuts[1:])]
            pcm = _pcm_session(g, pieces, prm)
            res = _flac_session(g, pieces, prm)
            _check_files(*res, pcm, 22050, f"{speeds} cuts {len(cuts) - 1}")
    finally:
        g.close()


@pytest.mark.parametrize("hz", (8000, 16000, 22050, 44100, 48000, ODD_RATE))
def test_rates(gpu, small_db, front_small, batch64, hz):
    plan = batch64[1]["mixed"]
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        g.set_output_rate(hz)
        pieces = [plan.select(range(0, 20)), plan.select(range(20, 64))]
        files = _check_files(*_flac_session(g, pieces, prm), _pcm_session(g, pieces, prm), hz, f"{hz} Hz")
        code = files[0][42 + 2] & 0xF
        assert code == {8000: 4, 16000: 5, 22050: 6, 44100: 9, 48000: 10}.get(hz, 13)
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
        _check_files(*_flac_session(g, [plan], prm), pcm, 22050, name)
    finally:
        g.close()


def test_empty_and_punctuation_only_texts(gpu, small_db, front_small):
    texts = ["", "...", "olá mundo", "!?", ", ;", ""]
    plan = front_small.plan(texts)
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        pcm = _pcm_session(g, [plan], prm)
        assert len(pcm[0]) == len(pcm[5]) == 0   # punctuation alone still yields its pause
        files = _check_files(*_flac_session(g, [plan], prm), pcm, 22050, "empty texts")
        assert len(files[0]) == len(files[5]) == 42
    finally:
        g.close()


def test_text_path_matches_the_session(gpu, pipe, small_db, front_small, batch64):
    texts, plans = batch64
    plan = plans["mixed"]
    speeds = np.asarray(plan.speed, np.float32)
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        out, off, nbytes, _, _ = _flac_session(g, [plan], prm)
        want = [out[int(off[u]):int(off[u]) + int(nbytes[u])].tobytes() for u in range(plan.n_utts)]
        batch = pipe.TextBatch(texts, speeds)
        cap = pipe.capacity_hint_flac(front_small, batch)
        assert cap >= g.flac_bound(plan)
        for piece_utts, threads in ((16, 1), (192, 3)):
            buf = np.zeros(cap, np.uint8)
            toff, tbytes, tcnt, used, tm = pipe.synth_texts_flac(front_small, g, batch, buf, piece_utts=piece_utts, threads=threads)
            assert used <= cap and tm.pieces >= 1
            for u in range(plan.n_utts):
                assert buf[int(toff[u]):int(toff[u]) + int(tbytes[u])].tobytes() == want[u], (piece_utts, threads, u)
    finally:
        g.close()


def test_full_batch_through_the_text_path(H, gpu, pipe, record_property):
    """BASELINE configs[2] (4096 utterances, ~200 characters, speed 1.0) through ctts_b200_synth_texts_flac: every
    file equals the oracle encoder on the PCM text path's output; 64 of them, the last 16 among them, decode to it."""
    db = H.synthetic_db()
    fr = H.front.Front(db, H.shipped_config(), H.NORM_CSV)
    texts = H.corpus.batch(4096, seed=1234)
    batch = pipe.TextBatch(texts)
    g = gpu.GpuSynth(db, 0)
    try:
        pcm_buf = np.zeros(pipe.capacity_hint(fr, batch), np.int16)
        poff, pcnt, _, _ = pipe.synth_texts(fr, g, batch, pcm_buf)
        out = np.zeros(pipe.capacity_hint_flac(fr, batch), np.uint8)
        off, nbytes, cnt, used, _ = pipe.synth_texts_flac(fr, g, batch, out)
        assert np.array_equal(cnt, pcnt)
        pcm = [pcm_buf[int(poff[u]):int(poff[u]) + int(pcnt[u])] for u in range(4096)]
        files = _check_files(out, off, nbytes, cnt, used, pcm, 22050, "configs[2]", decode=False)
        pick = sorted(set(np.random.default_rng(3).choice(4080, 48, replace=False).tolist()) | set(range(4080, 4096)))
        for u in pick:
            got, _ = F.decode(files[u])
            assert np.array_equal(got, pcm[u]), u
        pcm_bytes = 2 * int(pcnt.astype(np.int64).sum())
        flac_bytes = int(nbytes.astype(np.int64).sum())
        record_property("flac_bytes", flac_bytes)
        record_property("pcm_bytes", pcm_bytes)
        print(f"configs[2]: {flac_bytes} FLAC bytes for {pcm_bytes} PCM bytes, ratio {flac_bytes / pcm_bytes:.4f}")
        assert flac_bytes < pcm_bytes
    finally:
        g.close()


def test_too_small_capacity(gpu, small_db, front_small, batch64):
    plan = batch64[1]["speed1"]
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        pieces = [plan.select(range(a, a + 8)) for a in range(0, 64, 8)]
        _, off, nbytes, _, used = _flac_session(g, pieces, prm)
        # room for the first three pieces' files and a little more
        cap = int(off[24])
        L = gpu.lib()
        seen = []
        fn_t = C.CFUNCTYPE(None, C.c_void_p, C.c_uint32, C.c_uint32)
        cb = fn_t(lambda _u, b, e: seen.append((int(b), int(e))))
        out = np.zeros(cap + 8, np.uint8)
        h = C.c_void_p()
        g._check(L.ctts_gpu_session_begin_flac(g._h, C.byref(prm), out.ctypes.data, cap + 8, cb, None, C.byref(h)))
        o = np.zeros(64, np.uint64)
        b = np.zeros(64, np.uint32)
        c = np.zeros(64, np.uint32)
        rc = 0
        for i, p in enumerate(pieces):
            cp = p.as_c()
            rc = L.ctts_gpu_session_submit_flac(h, C.byref(cp), o[8 * i:].ctypes.data, b[8 * i:].ctypes.data, c[8 * i:].ctypes.data)
            if rc:
                break
        rc_end = L.ctts_gpu_session_end(h, None)
        assert (rc or rc_end) == ERR_BOUNDS
        # pieces before the one that does not fit may be handed over; that one and every later one are not
        assert seen == [(0, 8), (8, 16), (16, 24)][:len(seen)]
        # the context is usable afterwards, and the exact size is enough
        res = _flac_session(g, pieces, prm, cap=used)
        assert res[4] == used
    finally:
        g.close()


def test_pcm_and_flac_calls_do_not_mix(gpu, small_db, front_small, batch64):
    plan = batch64[1]["speed1"]
    prm = front_small.params()
    L = gpu.lib()
    g = gpu.GpuSynth(small_db, 0)
    try:
        cp = plan.as_c()
        o = np.zeros(64, np.uint64)
        b = np.zeros(64, np.uint32)
        c = np.zeros(64, np.uint32)
        h = C.c_void_p()
        pcm = np.zeros(1 << 22, np.int16)
        g._check(L.ctts_gpu_session_begin(g._h, C.byref(prm), pcm.ctypes.data, pcm.size, None, None, C.byref(h)))
        assert L.ctts_gpu_session_submit_flac(h, C.byref(cp), o.ctypes.data, b.ctypes.data, c.ctypes.data) == ERR_INVALID_ARG
        assert L.ctts_gpu_session_end(h, None) == 0
        out = np.zeros(g.flac_bound(plan), np.uint8)
        g._check(L.ctts_gpu_session_begin_flac(g._h, C.byref(prm), out.ctypes.data, out.size, None, None, C.byref(h)))
        assert L.ctts_gpu_session_submit(h, C.byref(cp), o.ctypes.data, c.ctypes.data) == ERR_INVALID_ARG
        assert L.ctts_gpu_session_submit_flac(h, C.byref(cp), o.ctypes.data, b.ctypes.data, c.ctypes.data) == 0
        used = C.c_uint64()
        assert L.ctts_gpu_session_end(h, C.byref(used)) == 0
        assert used.value == int((int(o[63]) + int(b[63]) + 15) // 16 * 16)
    finally:
        g.close()


def test_flac_header_symbols_are_exported(H, pipe):
    import test_abi
    names = test_abi._declared(os.path.join(H.ROOT, "include", "ctts_b200_flac.h"))
    assert names == ["ctts_b200_capacity_hint_flac", "ctts_b200_synth_texts_flac"]
    L = pipe.lib()
    for n in names:
        assert hasattr(L, n), n
    names = test_abi._declared(os.path.join(H.ROOT, "include", "ctts_gpu.h"))
    for n in ("ctts_gpu_session_begin_flac", "ctts_gpu_session_submit_flac", "ctts_gpu_flac_bound"):
        assert n in names and hasattr(H.importlib.import_module("2026-simple-c-tts_b200.gpu").lib(), n)


def test_pcm_path_is_unchanged_around_a_flac_session(gpu, small_db, front_small, batch64):
    plan = batch64[1]["mixed"]
    prm = front_small.params()
    g = gpu.GpuSynth(small_db, 0)
    try:
        pieces = [plan.select(range(0, 30)), plan.select(range(30, 64))]

        def pcm_bytes():
            n = plan.n_utts
            buf = np.zeros(sum(int(((g.bounds(p).astype(np.int64) + 7) // 8 * 8).sum()) for p in pieces), np.int16)
            off, cnt = g.synth_pieces(pieces, prm, buf)
            end = int(off[n - 1]) + (int(cnt[n - 1]) + 7) // 8 * 8
            return buf[:end].tobytes(), off.tobytes(), cnt.tobytes()
        before = pcm_bytes()
        _flac_session(g, pieces, prm)
        assert pcm_bytes() == before
    finally:
        g.close()


def test_command_line_writes_flac(H, small_db, tmp_path):
    b = H.importlib.import_module("2026-simple-c-tts_b200._build")
    exe = b.build_cli()
    shutil.copy(H.SHIPPED_YAML, tmp_path / "config.yaml")
    shutil.copy(H.NORM_CSV, tmp_path / "normalization.csv")
    (tmp_path / "voice.db").write_bytes(small_db)
    for name, extra in (("a", []), ("b", ["1.5", "16000"])):
        for ext in ("wav", "flac"):
            r = subprocess.run([exe, "synth", "voice.db", "olá mundo, bom dia", f"{name}.{ext}"] + extra, cwd=tmp_path,
                               capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
        wav = (tmp_path / f"{name}.wav").read_bytes()
        got, info = F.decode((tmp_path / f"{name}.flac").read_bytes())
        assert np.array_equal(got, np.frombuffer(wav[44:], "<i2"))
        assert info["sample_rate"] == int.from_bytes(wav[24:28], "little")
    (tmp_path / "t.tsv").write_text("1.0\tolá mundo\n1.5\tolá mundo\n1.0\t...\n", encoding="utf-8")
    for args in (["w"], ["f", "22050", "flac"]):
        r = subprocess.run([exe, "synth-batch", "voice.db", "t.tsv"] + args, cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    for u in range(3):
        wav = (tmp_path / "w" / f"{u:06d}.wav").read_bytes()
        got, _ = F.decode((tmp_path / "f" / f"{u:06d}.flac").read_bytes())
        assert np.array_equal(got, np.frombuffer(wav[44:], "<i2")), u
