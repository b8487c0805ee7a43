"""GPU tests of the true-peak ceiling of the loudness normalization (ctts_gpu_set_loudness_true_peak, DESIGN.md 3.6):
on every entry point the device's true peak P equals the oracle's (tests/true_peak_oracle.c) bit for bit, its G and its
output equal the oracle's and its L agrees to 1e-6 LU, applied to the PCM the context delivers with the stage off.
Constructed signals put the peak at the ends of an utterance and at the true-peak kernel's tile boundaries; a
sample-peak setting made after a true-peak one is exactly the sample-peak stage; bad calls are rejected.

Run on a B200 with:  python -m pytest tests/test_gpu_true_peak.py -m gpu
"""
import ctypes as Ct
import shutil
import subprocess

import numpy as np
import pytest

import edge_voices as E
import flac_codec as F
import loudness_oracle as O
import true_peak_oracle as TP
import resample_oracle as R
from test_gpu_loudness import _check_ld, _check_pcm, _slices, _up8, batch64  # noqa: F401  (batch64: fixture)
from test_true_peak import square4

pytestmark = pytest.mark.gpu

ERR_INVALID_ARG = -1
SETTINGS = ((-16.0, -1.0), (-23.0, -2.0))
TILE = 2048          # LD_TP_TILE: positions per ld_true_peak_kernel CTA
EDGE = TILE - 6      # the first position of tile 1 (tile 0 starts at position -6)


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.fixture(scope="module")
def pipe(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.pipeline")


def _tp_ctx(gpu, db, hz, T=0.0, C=-1.0, true_peak=True):
    g = gpu.GpuSynth(db, 0)
    g.set_output_rate(hz)
    if T:
        g.set_loudness(T, C, true_peak=true_peak)
    return g


def _oracle(xs, hz, T, C):
    """([(y, L, G)], [P]) of the oracle with a true-peak ceiling."""
    w = [TP.normalize(x, hz, T, C) for x in xs]
    return [(y, L, G) for y, L, G, _ in w], np.array([P for _, _, _, P in w], np.float32)


def _check_resident(rp, want, peaks, T, what):
    lufs, gain = rp.loudness()
    ties = _check_ld(lufs, gain, want, T, what)
    got = rp.true_peak()
    assert got.dtype == np.float32 and len(got) == len(peaks)
    bad = np.nonzero(got.view(np.uint32) != peaks.view(np.uint32))[0]
    assert not len(bad), f"{what}: P differs at {bad[:5]}: {got[bad[:5]]} vs the oracle's {peaks[bad[:5]]}"
    _check_pcm(rp.utterances(), want, ties, what)
    return ties


@pytest.mark.parametrize("T,C", SETTINGS)
@pytest.mark.parametrize("hz", (8000, 11025, 16000, 22050, 48000))
def test_every_entry_point_matches_the_oracle(gpu, pipe, small_db, front_small, batch64, hz, T, C):
    texts, speeds, plan, prm, native = batch64
    want, peaks = _oracle([R.resample(x, hz) for x in native], hz, T, C)
    n = plan.n_utts
    g = _tp_ctx(gpu, small_db, hz, T, C)
    try:
        bounds = g.bounds(plan).astype(np.int64)
        rp = g.create_plan(plan, prm)
        for run in range(2):
            rp.run()
            ties = _check_resident(rp, want, peaks, T, f"{hz} {T} resident run {run}")
        rp.close()
        pcm, off, cnt = g.synth_batch(plan, prm)
        _check_pcm(_slices(pcm, off, cnt), want, ties, f"{hz} {T} synth_batch")
        cap = int(_up8(bounds).sum())
        buf = np.zeros(cap, np.int16)
        poff, pcnt, _ = g.synth_batch_packed(plan, prm, buf)
        _check_pcm(_slices(buf, poff, pcnt), want, ties, f"{hz} {T} packed")
        cuts = [0, 1, 9, 9, 30, 31, 50, 64]
        pieces = [plan.select(range(a, b)) for a, b in zip(cuts[:-1], cuts[1:])]
        buf = np.zeros(cap + 64, np.int16)
        soff, scnt = g.synth_pieces(pieces, prm, buf)
        _check_pcm(_slices(buf, soff, scnt), want, ties, f"{hz} {T} session")
        out = np.zeros(sum(g.flac_bound(p) for p in pieces), np.uint8)
        foff, fbytes, _, _ = g.synth_pieces_flac(pieces, prm, out)
        dec = [F.decode(out[int(foff[u]):int(foff[u]) + int(fbytes[u])].tobytes())[0] for u in range(n)]
        _check_pcm(dec, want, ties, f"{hz} {T} FLAC session")
        batch = pipe.TextBatch(texts, speeds)
        tbuf = np.zeros(pipe.capacity_hint(front_small, batch, hz), np.int16)
        toff, tcnt, _, _ = pipe.synth_texts(front_small, g, batch, tbuf)
        _check_pcm(_slices(tbuf, toff, tcnt), want, ties, f"{hz} {T} synth_texts")
    finally:
        g.close()
    ctxs = [_tp_ctx(gpu, small_db, hz, T, C) for _ in range(3)]
    try:
        mpcm, moff, mcnt, shard = gpu.multi_synth_batch(ctxs, plan, prm)
        assert len(set(shard.tolist())) == 3
        _check_pcm(_slices(mpcm, moff, mcnt), want, ties, f"{hz} {T} multi")
    finally:
        for c in ctxs:
            c.close()


# ---------------------------------------------------------------------------------- constructed signals

SR = 22050
QUIET_LEN = SR   # one second: L is defined


def _quiet(rng, n):
    return E.harmonic(rng, n, peak=400.0)


def _low_square_setting():
    """(T, C, amplitude) where the period-4 square's true peak limits G and its sample peak would not."""
    x = square4(QUIET_LEN, 300)
    for C in (-20.0, -12.0, -6.0):
        for T in np.arange(-40.0, -5.0, 0.25):
            L = O.lufs(x, SR)
            _, _, G, P = TP.normalize(x, SR, float(T), C)
            Gs = O.gain(L, float(T), C, 300)
            if G < Gs and Gs == int(O.table()[int(np.floor(100 * (np.float32(T) - L) + 0.5)) + O.K_MAX]):
                return float(T), C
    raise AssertionError("no setting where only the true peak limits the square")


def tp_signals(seed: int = 41):
    """(case, signal) pairs at 22 050 Hz (the voice's own rate: the signal reaches the stage unchanged)."""
    rng = np.random.default_rng(seed)
    out = [("square4_full", square4(QUIET_LEN)), ("square4_low", square4(QUIET_LEN, 300))]
    for at in ("first", "last"):
        x = _quiet(rng, QUIET_LEN)
        x[0 if at == "first" else -1] = -32768
        out.append((f"peak_{at}", x))
    for d in (-6, -1, 0, 1, 6):
        for edge in (EDGE, 2 * TILE + EDGE):
            x = _quiet(rng, 5 * TILE)   # 464 ms: L is defined
            x[edge + d - 1:edge + d + 1] = (32767, -32767)   # an over of about +2 dB centred at the boundary +- d
            out.append((f"edge{edge}{d:+d}", x))
    for n in range(14):
        out.append((f"len{n}", rng.integers(-32768, 32768, n).astype(np.int16)))
    for k in (1, 2, 10):
        for d in (-1, 0, 1):
            n = k * TILE - 12 + d   # positions -6 .. n + 5 fill k tiles exactly, one more, one less
            out.append((f"tiles{k}{d:+d}", np.roll(square4(n, 20000), int(rng.integers(4)))))
            x = _quiet(rng, k * TILE + d)
            x[-1] = 32767
            out.append((f"len{k}x{TILE}{d:+d}", x))
    short = square4(1000)   # under 400 ms: L undefined, unity G, P still reported
    out.append(("undefined", short))
    return out


@pytest.fixture(scope="module")
def tp_family():
    sig = tp_signals()
    return E.family_signals("true_peak", [x for _, x in sig]), [n for n, _ in sig]


def test_constructed_signals(gpu, tp_family):
    fam, names = tp_family
    plan, prm = fam.plan(), fam.prm()
    xs = fam.info["signals"]
    Tl, Cl = _low_square_setting()
    low = names.index("square4_low")
    und = names.index("undefined")
    for T, C in SETTINGS + ((Tl, Cl),):
        want, peaks = _oracle(xs, SR, T, C)
        if (T, C) == (Tl, Cl):
            L = want[low][1]
            assert want[low][2] < O.gain(L, T, C, 300), "the low square must be limited by its true peak"
        assert want[und][2] == O.UNITY and not np.isfinite(want[und][1]) and peaks[und] > 32767
        g = _tp_ctx(gpu, fam.db, SR, T, C)
        try:
            rp = g.create_plan(plan, prm)
            for run in range(2):
                rp.run()
                ties = _check_resident(rp, want, peaks, T, f"signals T {T} C {C} run {run}")
            rp.close()
            pcm, off, cnt = g.synth_batch(plan, prm)
            _check_pcm(_slices(pcm, off, cnt), want, ties, f"signals T {T} C {C} synth_batch")
        finally:
            g.close()


# ---------------------------------------------------------------------------------- settings

def _run(g, plan, prm):
    rp = g.create_plan(plan, prm)
    rp.run()
    r = (rp.info().kernel_launches, rp.counts().tobytes(), b"".join(x.tobytes() for x in rp.utterances()))
    rp.close()
    return r


def test_settings(gpu, small_db, batch64):
    _, _, plan, prm, native = batch64
    hz, T, C = 16000, -16.0, -1.0
    xs = [R.resample(x, hz) for x in native]
    never = _tp_ctx(gpu, small_db, hz, T, C, true_peak=False)
    g = _tp_ctx(gpu, small_db, hz, T, C)
    try:
        # a sample-peak setting made after a true-peak one is the sample-peak stage: bytes and launches
        base = _run(never, plan, prm)
        tp = _run(g, plan, prm)
        assert tp[0] == base[0] + 1
        g.set_loudness(T, C)
        assert _run(g, plan, prm) == base
        # switching kinds on one context, and a plan keeps its kind
        g.set_loudness(-23.0, -2.0, true_peak=True)
        rp = g.create_plan(plan, prm)
        g.set_loudness(-23.0, -2.0)
        g.set_output_rate(8000)
        rp.run()
        want, peaks = _oracle(xs, hz, -23.0, -2.0)
        _check_resident(rp, want, peaks, -23.0, "kept true-peak plan")
        rp.close()
        pcm, off, cnt = g.synth_batch(plan, prm)
        w8 = [O.normalize(R.resample(x, 8000), 8000, -23.0, -2.0) for x in native]
        _check_pcm(_slices(pcm, off, cnt), w8, set(), "sample peak at 8 kHz")
        g.set_loudness(-23.0, -2.0, true_peak=True)   # follows the rate
        want8, peaks8 = _oracle([R.resample(x, 8000) for x in native], 8000, -23.0, -2.0)
        rp = g.create_plan(plan, prm)
        rp.run()
        _check_resident(rp, want8, peaks8, -23.0, "true peak at 8 kHz")
        rp.close()
    finally:
        never.close()
        g.close()


def test_errors(gpu, small_db, batch64):
    _, _, plan, prm, _ = batch64
    lib = gpu.lib()
    g = _tp_ctx(gpu, small_db, 16000, -16.0, -1.0)
    gs = _tp_ctx(gpu, small_db, 16000, -16.0, -1.0, true_peak=False)
    try:
        pcm0, off0, cnt0 = g.synth_batch(plan, prm)
        for T, C in [(-16.0, 0.1), (-16.0, -20.5), (-16.0, float("nan")), (-16.0, float("inf")), (-4.0, -1.0),
                     (float("nan"), -1.0)]:
            assert lib.ctts_gpu_set_loudness_true_peak(g._h, T, C) == ERR_INVALID_ARG, (T, C)
        h = Ct.c_void_p()
        buf = np.zeros(1024, np.int16)
        assert lib.ctts_gpu_session_begin(g._h, Ct.byref(prm), buf.ctypes.data, buf.size, None, None, Ct.byref(h)) == 0
        assert lib.ctts_gpu_set_loudness_true_peak(g._h, -23.0, -1.0) == ERR_INVALID_ARG
        assert lib.ctts_gpu_session_end(h, None) == 0
        pcm1, off1, cnt1 = g.synth_batch(plan, prm)
        assert np.array_equal(cnt0, cnt1)
        assert all(np.array_equal(a, b) for a, b in zip(_slices(pcm0, off0, cnt0), _slices(pcm1, off1, cnt1)))
        for mix in ([g, gs], [gs, g]):
            with pytest.raises(gpu.GpuError):
                gpu.multi_synth_batch(mix, plan, prm)
        rp = gs.create_plan(plan, prm)
        rp.run()
        with pytest.raises(gpu.GpuError):
            rp.true_peak()
        rp.close()
    finally:
        g.close()
        gs.close()


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
    want = {k: TP.normalize(R.resample(oracle_small.synth(prm, plan.utt_ops(u), PAIRS[k][1])[0], hz), hz, T, C)
            for k, u in first.items()}
    g = _tp_ctx(gpu, small_db, hz, T, C)
    try:
        rp = g.create_plan(plan, prm)
        rp.run()
        cnt, off = rp.counts().astype(np.int64), rp.out_offsets().astype(np.int64)
        pcm = rp.read_pcm(0, int(off[-1]))
        lufs, gain = rp.loudness()
        peaks = rp.true_peak()
        for u in list(range(0, 200)) + list(range(65400, 65700)) + list(range(N_BIG - 300, N_BIG)):
            y, L, G, P = want[int(pick[u])]
            assert peaks[u] == np.float32(P), (u, peaks[u], P)
            ties = _check_ld(lufs[u:u + 1], gain[u:u + 1], [(y, L, G)], T, f"big utt {u}")
            if not ties:
                assert np.array_equal(pcm[off[u]:off[u] + cnt[u]], y), u
    finally:
        g.close()


def test_command_line(H, gpu, pipe, small_db, front_small, tmp_path):
    """dbtp= next to lufs=: the WAV samples are the oracle's, applied to the text path's output with the stage off."""
    b = H.importlib.import_module("2026-simple-c-tts_b200._build")
    exe = b.build_cli()
    shutil.copy(H.SHIPPED_YAML, tmp_path / "config.yaml")
    shutil.copy(H.NORM_CSV, tmp_path / "normalization.csv")
    (tmp_path / "voice.db").write_bytes(small_db)
    texts = ["Bom dia, como vai? São 1234 casas, não é verdade?", "olá mundo"]
    g = _tp_ctx(gpu, small_db, 22050)
    try:
        batch = pipe.TextBatch(texts, [1.0, 1.0])
        tbuf = np.zeros(pipe.capacity_hint(front_small, batch, 22050), np.int16)
        toff, tcnt, _, _ = pipe.synth_texts(front_small, g, batch, tbuf)
        want = [TP.normalize(x, 22050, -16.0, -2.0)[0] for x in _slices(tbuf, toff, tcnt)]
    finally:
        g.close()
    r = subprocess.run([exe, "synth", "voice.db", texts[0], "o.wav", "1.0", "22050", "dbtp=-2", "lufs=-16"], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(np.frombuffer((tmp_path / "o.wav").read_bytes()[44:], dtype="<i2"), want[0])
    (tmp_path / "t.tsv").write_text("".join(f"1.0\t{t}\n" for t in texts), encoding="utf-8")
    r = subprocess.run([exe, "synth-batch", "voice.db", "t.tsv", "out", "22050", "lufs=-16", "dbtp=-2"], cwd=tmp_path,
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    for u in range(2):
        raw = (tmp_path / "out" / f"{u:06d}.wav").read_bytes()
        assert np.array_equal(np.frombuffer(raw[44:], dtype="<i2"), want[u]), u
    for bad in (["dbtp=-2"], ["lufs=-16", "dbtp=1"], ["lufs=-16", "dbtp=x"], ["dbtp=-1", "lufs=-16", "dbtp=-2"]):
        r = subprocess.run([exe, "synth", "voice.db", texts[1], "bad.wav", "1.0", "22050"] + bad, cwd=tmp_path,
                           capture_output=True, text=True)
        assert r.returncode != 0 and not (tmp_path / "bad.wav").exists(), bad
