"""GPU tests of the loudness normalization (ctts_gpu_set_loudness, DESIGN.md 3.6): on every entry point the device's L
agrees with the oracle (tests/loudness_oracle.c) to 1e-6 LU, its G and its output equal the oracle's, applied to the
PCM the context delivers with the stage off (itself pinned bit for bit by the resample and parity suites).  Off
leaves every path as it was; bad settings are rejected.

Run on a B200 with:  python -m pytest tests/test_gpu_loudness.py -m gpu
"""
import math
import shutil
import subprocess
import warnings

import numpy as np
import pytest

import edge_voices as E
import flac_codec as F
import loudness_oracle as O
import resample_oracle as R

pytestmark = pytest.mark.gpu

ERR_INVALID_ARG = -1
SETTINGS = ((-16.0, -1.0), (-23.0, -3.0))


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.fixture(scope="module")
def pipe(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.pipeline")


def _up8(v):
    return (np.asarray(v, np.int64) + 7) // 8 * 8


def _assert_same(got, want, what=""):
    assert len(got) == len(want), f"{what}: length {len(got)} != {len(want)}"
    if not np.array_equal(got, want):
        d = np.nonzero(got != want)[0]
        raise AssertionError(f"{what}: {len(d)} of {len(want)} samples differ, first at {d[:5]}")


def _oracle(xs, hz, T, C):
    """[(y, L, G)] of the oracle on every utterance."""
    return [O.normalize(x, hz, T, C) for x in xs]


def _ties(want, T):
    """Utterances whose 100 (T - L) lies within 1e-4 of a half-integer: reported, never compared silently."""
    t = [u for u, (_, L, _) in enumerate(want) if O.near_tie(L, T)]
    if t:
        warnings.warn(f"loudness: utterances {t} are within 1e-4 of a rounding tie of k; their gain is not compared")
    return set(t)


def _check_ld(lufs, gain, want, T, what):
    ties = _ties(want, T)
    for u, (_, L, G) in enumerate(want):
        if math.isinf(L):
            assert lufs[u] == -np.inf, f"{what}: utterance {u}: L {lufs[u]} where the oracle's is undefined"
        else:
            assert abs(lufs[u] - L) <= 1e-6, f"{what}: utterance {u}: L {lufs[u]!r} vs the oracle's {L!r}"
        if u not in ties:
            assert int(gain[u]) == G, f"{what}: utterance {u}: G {int(gain[u])} vs the oracle's {G}"
    return ties


def _check_pcm(got, want, ties, what):
    for u, (y, _, _) in enumerate(want):
        if u not in ties:
            _assert_same(got[u], y, f"{what} utt {u}")


@pytest.fixture(scope="module")
def batch64(H, front_small, oracle_small):
    """64 utterances of the small voice, mixed speeds, with the oracle's native PCM."""
    texts = H.corpus.batch(61, seed=4242, target_chars=90) + ["", "olá mundo", "São 1234 casas, não é?"]
    speeds = list(H.corpus.mixed_speeds(64, seed=17))
    speeds[::3] = [1.0] * len(speeds[::3])
    plan = front_small.plan(texts, speeds)
    prm = front_small.params()
    native = [oracle_small.synth(prm, plan.utt_ops(u), float(speeds[u]))[0] for u in range(plan.n_utts)]
    return texts, speeds, plan, prm, native


def _ctx(gpu, db, hz, T=0.0, C=-1.0):
    g = gpu.GpuSynth(db, 0)
    g.set_output_rate(hz)
    if T:
        g.set_loudness(T, C)
    return g


def _slices(buf, off, cnt):
    return [buf[int(off[u]):int(off[u]) + int(cnt[u])] for u in range(len(cnt))]


@pytest.mark.parametrize("T,C", SETTINGS)
@pytest.mark.parametrize("hz", (22050, 16000, 8000, 48000))
def test_every_entry_point_matches_the_oracle(gpu, pipe, small_db, front_small, batch64, hz, T, C):
    texts, speeds, plan, prm, native = batch64
    want = _oracle([R.resample(x, hz) for x in native], hz, T, C)
    assert any(G != O.UNITY for _, _, G in want)
    n = plan.n_utts
    g = _ctx(gpu, small_db, hz, T, C)
    try:
        bounds = g.bounds(plan).astype(np.int64)
        rp = g.create_plan(plan, prm)
        for run in range(2):
            rp.run()
            lufs, gain = rp.loudness()
            ties = _check_ld(lufs, gain, want, T, f"{hz} {T} resident run {run}")
            _check_pcm(rp.utterances(), want, ties, f"{hz} {T} resident run {run}")
        rp.close()
        pcm, off, cnt = g.synth_batch(plan, prm)
        _check_pcm(_slices(pcm, off, cnt), want, ties, f"{hz} {T} synth_batch")
        cap = int(_up8(bounds).sum())
        buf = np.zeros(cap, np.int16)
        poff, pcnt, _ = g.synth_batch_packed(plan, prm, buf)
        _check_pcm(_slices(buf, poff, pcnt), want, ties, f"{hz} {T} packed")
        got = [None] * n

        def on_chunk(pcm_, off_, cnt_, a, b):
            for u in range(a, b):
                got[u] = pcm_[int(off_[u]):int(off_[u]) + int(cnt_[u])].copy()
        g.synth_batch_stream(plan, prm, on_chunk)
        _check_pcm(got, want, ties, f"{hz} {T} stream")
        cuts = [0, 1, 9, 9, 30, 31, 50, 64]
        pieces = [plan.select(range(a, b)) for a, b in zip(cuts[:-1], cuts[1:])]
        buf = np.zeros(cap + 64, np.int16)
        soff2, scnt2 = g.synth_pieces(pieces, prm, buf)
        _check_pcm(_slices(buf, soff2, scnt2), want, ties, f"{hz} {T} session")
        out = np.zeros(sum(g.flac_bound(p) for p in pieces), np.uint8)
        foff, fbytes, fcnt, _ = g.synth_pieces_flac(pieces, prm, out)
        dec = [F.decode(out[int(foff[u]):int(foff[u]) + int(fbytes[u])].tobytes())[0] for u in range(n)]
        _check_pcm(dec, want, ties, f"{hz} {T} FLAC session")
        batch = pipe.TextBatch(texts, speeds)
        tbuf = np.zeros(pipe.capacity_hint(front_small, batch, hz), np.int16)
        toff, tcnt, _, _ = pipe.synth_texts(front_small, g, batch, tbuf)
        _check_pcm(_slices(tbuf, toff, tcnt), want, ties, f"{hz} {T} synth_texts")
    finally:
        g.close()
    ctxs = [_ctx(gpu, small_db, hz, T, C) for _ in range(3)]
    try:
        mpcm, moff, mcnt, shard = gpu.multi_synth_batch(ctxs, plan, prm)
        assert len(set(shard.tolist())) == 3
        _check_pcm(_slices(mpcm, moff, mcnt), want, ties, f"{hz} {T} multi")
    finally:
        for c in ctxs:
            c.close()


EDGE = ("amplitude_rms0", "amplitude_rms3000", "tiny_stretch", "short_units")


@pytest.mark.parametrize("hz", (8000, 16000, 22050))
@pytest.mark.parametrize("name", EDGE)
def test_edge_voices(gpu, name, hz):
    """Full-scale, rms < 1, gain-clamped and large-DC units; 0-769-sample and all-zero utterances; very short units."""
    fam = E.family(name)
    plan, prm = fam.plan(), fam.prm()
    xs = [R.resample(x, hz) for x in fam.expected()]
    for T, C in SETTINGS:
        want = _oracle(xs, hz, T, C)
        g = _ctx(gpu, fam.db, hz, T, C)
        try:
            rp = g.create_plan(plan, prm)
            rp.run()
            lufs, gain = rp.loudness()
            ties = _check_ld(lufs, gain, want, T, f"{name} {hz}")
            got = rp.utterances()
            _check_pcm(got, want, ties, f"{name} {hz}")
            A = O.ceiling(C)
            for u, (x, (_, L, _)) in enumerate(zip(xs, want)):
                if math.isinf(L):
                    _assert_same(got[u], x, f"{name} {hz} undefined L, utt {u}")
                elif len(x):
                    assert np.abs(got[u].astype(np.int32)).max() <= A, f"{name} {hz} utt {u} passes the ceiling"
        finally:
            g.close()


def test_off_is_unchanged(gpu, small_db, batch64):
    _, _, plan, prm, _ = batch64
    for hz in (22050, 16000):
        runs = []
        for setting in ("never", "reset"):
            g = _ctx(gpu, small_db, hz)
            try:
                if setting == "reset":
                    g.set_loudness(-16.0, -1.0)
                    g.set_loudness(0.0)
                rp = g.create_plan(plan, prm)
                rp.run()
                cnt = rp.counts()
                runs.append((rp.info().kernel_launches, cnt.tobytes(), b"".join(x.tobytes() for x in rp.utterances())))
                with pytest.raises(gpu.GpuError):
                    rp.loudness()
                rp.close()
                pcm, off, cnt = g.synth_batch(plan, prm)
                runs[-1] += (b"".join(x.tobytes() for x in _slices(pcm, off, cnt)),)
            finally:
                g.close()
        assert runs[0] == runs[1]
        g = _ctx(gpu, small_db, hz, -16.0)
        try:
            on = g.create_plan(plan, prm).info().kernel_launches
        finally:
            g.close()
        assert on == runs[0][0] + 5


def test_errors(gpu, small_db, batch64):
    _, _, plan, prm, native = batch64
    lib = gpu.lib()
    g = _ctx(gpu, small_db, 16000, -16.0, -1.0)
    g2 = _ctx(gpu, small_db, 16000, -23.0, -1.0)
    g3 = _ctx(gpu, small_db, 16000)
    try:
        pcm0, off0, cnt0 = g.synth_batch(plan, prm)
        bad = [(math.nan, -1.0), (math.inf, -1.0), (-math.inf, -1.0), (-60.5, -1.0), (-4.9, -1.0), (3.0, -1.0),
               (-16.0, math.nan), (-16.0, math.inf), (-16.0, -math.inf), (-16.0, 0.1), (-16.0, -20.5), (0.0, math.nan)]
        for T, C in bad:
            assert lib.ctts_gpu_set_loudness(g._h, T, C) == ERR_INVALID_ARG, (T, C)
        # a call while a session is open
        import ctypes as Ct
        h = Ct.c_void_p()
        buf = np.zeros(1024, np.int16)
        assert lib.ctts_gpu_session_begin(g._h, Ct.byref(prm), buf.ctypes.data, buf.size, None, None, Ct.byref(h)) == 0
        assert lib.ctts_gpu_set_loudness(g._h, -23.0, -1.0) == ERR_INVALID_ARG
        assert lib.ctts_gpu_set_loudness(g._h, 0.0, -1.0) == ERR_INVALID_ARG
        assert lib.ctts_gpu_session_end(h, None) == 0
        pcm1, off1, cnt1 = g.synth_batch(plan, prm)
        assert np.array_equal(cnt0, cnt1)
        for u in range(plan.n_utts):
            _assert_same(pcm1[off1[u]:off1[u] + cnt1[u]], pcm0[off0[u]:off0[u] + cnt0[u]], f"after rejected settings, utt {u}")
        # mixed settings across contexts
        for mix in ([g, g2], [g, g3], [g3, g]):
            with pytest.raises(gpu.GpuError):
                gpu.multi_synth_batch(mix, plan, prm)
        # a plan keeps its setting after the context changes
        rp = g.create_plan(plan, prm)
        g.set_loudness(-30.0, -6.0)
        g.set_output_rate(8000)
        rp.run()
        want = _oracle([R.resample(x, 16000) for x in native], 16000, -16.0, -1.0)
        lufs, gain = rp.loudness()
        ties = _check_ld(lufs, gain, want, -16.0, "kept setting")
        _check_pcm(rp.utterances(), want, ties, "kept setting")
        rp.close()
        # and the context now runs the new setting at the new rate
        want = _oracle([R.resample(x, 8000) for x in native], 8000, -30.0, -6.0)
        pcm, off, cnt = g.synth_batch(plan, prm)
        _check_pcm(_slices(pcm, off, cnt), want, _ties(want, -30.0), "new setting at 8 kHz")
    finally:
        for c in (g, g2, g3):
            c.close()


def test_full_batch_at_22050(H, gpu):
    """BASELINE configs[2] (4096 utterances): every utterance is held to the ceiling, every one that is neither
    peak-limited nor undefined measures T +- 0.05 LU by the oracle, and 64 equal the oracle bit for bit."""
    db = H.synthetic_db()
    fr = H.front.Front(db, H.shipped_config(), H.NORM_CSV)
    prm = fr.params()
    plan = fr.plan(H.corpus.batch(4096, seed=1234))
    hz, T, C = 22050, -16.0, -1.0
    A = O.ceiling(C)
    g = gpu.GpuSynth(db, 0)
    try:
        rp = g.create_plan(plan, prm)
        rp.run()
        cnt0, off0 = rp.counts().astype(np.int64), rp.out_offsets().astype(np.int64)
        x_all = rp.read_pcm(0, int(off0[-1]))
        rp.close()
        g.set_loudness(T, C)
        rp = g.create_plan(plan, prm)
        rp.run()
        cnt, off = rp.counts().astype(np.int64), rp.out_offsets().astype(np.int64)
        assert np.array_equal(cnt, cnt0) and np.array_equal(off, off0)
        y_all = rp.read_pcm(0, int(off[-1]))
        lufs, gain = rp.loudness()
        pick = set(np.random.default_rng(5).choice(4096, 64, replace=False).tolist())
        for u in range(plan.n_utts):
            x = x_all[off[u]:off[u] + cnt[u]]
            y = y_all[off[u]:off[u] + cnt[u]]
            assert not len(y) or np.abs(y.astype(np.int32)).max() <= A, u
            if u in pick:
                want = [O.normalize(x, hz, T, C)]
                ties = _check_ld(lufs[u:u + 1], gain[u:u + 1], want, T, f"configs[2] utt {u}")
                if not ties:
                    _assert_same(y, want[0][0], f"configs[2] utt {u}")
            peak = int(np.abs(x.astype(np.int32)).max()) if len(x) else 0
            limited = peak and int(gain[u]) == A * 65536 // peak
            clamped = np.isfinite(lufs[u]) and abs(100 * (T - lufs[u])) > 7999
            if np.isfinite(lufs[u]) and not limited and not clamped:
                assert abs(O.lufs(y, hz) - T) <= 0.05, (u, lufs[u], int(gain[u]))
    finally:
        g.close()


N_BIG = 80000
PAIRS = [("olá", 1.5), ("bom dia", 0.75), ("casa", 1.25), ("São 1234 casas, não é?", 1.0), ("não", 2.0),
         ("Bom dia, como vai? Olá mundo, bom dia.", 1.0), ("olá dia", 1.0)]


def test_more_than_65535_utterances(gpu, small_db, front_small, oracle_small, monkeypatch):
    monkeypatch.setenv("CTTS_GPU_CHUNK_SAMPLES", str(1 << 40))   # read at init: one piece holds the whole batch
    hz, T, C = 16000, -16.0, -1.0
    pick = np.arange(N_BIG) % len(PAIRS)
    plan = front_small.plan([PAIRS[k][0] for k in pick], [PAIRS[k][1] for k in pick])
    prm = front_small.params()
    first = {int(k): int(np.argmax(pick == k)) for k in np.unique(pick)}
    want = {k: O.normalize(R.resample(oracle_small.synth(prm, plan.utt_ops(u), PAIRS[k][1])[0], hz), hz, T, C)
            for k, u in first.items()}
    assert any(np.isfinite(w[1]) for w in want.values())
    g = _ctx(gpu, small_db, hz, T, C)
    try:
        rp = g.create_plan(plan, prm)
        rp.run()
        cnt, off = rp.counts().astype(np.int64), rp.out_offsets().astype(np.int64)
        pcm = rp.read_pcm(0, int(off[-1]))
        lufs, gain = rp.loudness()
        check = list(range(0, 200)) + list(range(65400, 65700)) + list(range(N_BIG - 300, N_BIG))
        for u in check:
            y, L, G = want[int(pick[u])]
            ties = _check_ld(lufs[u:u + 1], gain[u:u + 1], [(y, L, G)], T, f"big utt {u}")
            if not ties:
                _assert_same(pcm[off[u]:off[u] + cnt[u]], y, f"big utt {u}")
    finally:
        g.close()


def test_command_line(H, small_db, gpu, pipe, front_small, tmp_path):
    b = H.importlib.import_module("2026-simple-c-tts_b200._build")
    exe = b.build_cli()
    shutil.copy(H.SHIPPED_YAML, tmp_path / "config.yaml")
    shutil.copy(H.NORM_CSV, tmp_path / "normalization.csv")
    (tmp_path / "voice.db").write_bytes(small_db)
    texts = ["Bom dia, como vai? São 1234 casas, não é verdade?", "olá mundo"]
    g = _ctx(gpu, small_db, 22050, -16.0, -1.0)
    try:
        batch = pipe.TextBatch(texts, [1.0, 1.0])
        tbuf = np.zeros(pipe.capacity_hint(front_small, batch, 22050), np.int16)
        toff, tcnt, _, _ = pipe.synth_texts(front_small, g, batch, tbuf)
        lib_pcm = _slices(tbuf, toff, tcnt)
    finally:
        g.close()
    r = subprocess.run([exe, "synth", "voice.db", texts[0], "o.wav", "1.0", "22050", "lufs=-16"], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = (tmp_path / "o.wav").read_bytes()
    assert np.array_equal(np.frombuffer(raw[44:], dtype="<i2"), lib_pcm[0])
    (tmp_path / "t.tsv").write_text("".join(f"1.0\t{t}\n" for t in texts), encoding="utf-8")
    r = subprocess.run([exe, "synth-batch", "voice.db", "t.tsv", "out", "22050", "lufs=-16"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for u in range(2):
        raw = (tmp_path / "out" / f"{u:06d}.wav").read_bytes()
        assert np.array_equal(np.frombuffer(raw[44:], dtype="<i2"), lib_pcm[u]), u
    r = subprocess.run([exe, "synth", "voice.db", texts[1], "bad.wav", "1.0", "22050", "lufs=-3"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and not (tmp_path / "bad.wav").exists()
