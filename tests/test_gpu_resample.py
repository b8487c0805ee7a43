"""GPU tests of the output-rate conversion (ctts_gpu_set_output_rate, DESIGN.md 3.4): every entry point delivers,
bit for bit, the oracle's synthesis followed by the oracle's resampler (tests/resample_oracle.c); counts, bounds and
capacities are in output-rate samples; 22 050 Hz leaves every path as it was.

Run on a B200 with:  python -m pytest tests/test_gpu_resample.py -m gpu
"""
import shutil
import struct
import subprocess

import numpy as np
import pytest

import edge_voices as E
import resample_oracle as R

pytestmark = pytest.mark.gpu

RATES = (8000, 11025, 16000, 24000, 44100, 48000)
ERR_INVALID_ARG = -1


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
        raise AssertionError(f"{what}: {len(d)} of {len(want)} samples differ, first at {d[:5]}, "
                             f"max |d| {np.abs(got.astype(int) - want.astype(int)).max()}")


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


def _ctx(gpu, db, hz):
    g = gpu.GpuSynth(db, 0)
    g.set_output_rate(hz)
    return g


@pytest.mark.parametrize("hz", RATES)
def test_every_entry_point_matches_the_oracle(H, gpu, pipe, small_db, front_small, batch64, hz):
    texts, speeds, plan, prm, native = batch64
    want = [R.resample(x, hz) for x in native]
    n = plan.n_utts
    g = _ctx(gpu, small_db, hz)
    try:
        bounds = g.bounds(plan).astype(np.int64)
        L, M = R.ratio(hz)
        # synth_batch with caller slots (sized by the output-rate bounds)
        pcm, off, cnt = g.synth_batch(plan, prm)
        assert (cnt.astype(np.int64) <= bounds).all()
        for u in range(n):
            _assert_same(pcm[int(off[u]):int(off[u]) + int(cnt[u])], want[u], f"{hz} synth_batch utt {u}")
        # synth_batch_packed, with exactly the capacity the bounds promise
        cap = int(_up8(bounds).sum())
        buf = np.zeros(cap, np.int16)
        poff, pcnt, used = g.synth_batch_packed(plan, prm, buf)
        assert used == int(_up8(pcnt).sum()) <= cap
        for u in range(n):
            _assert_same(buf[int(poff[u]):int(poff[u]) + int(pcnt[u])], want[u], f"{hz} packed utt {u}")
        # a resident plan, run twice
        rp = g.create_plan(plan, prm)
        assert rp.out_samples == int(g.layout(plan)[-1])
        for run in range(2):
            rp.run()
            for u, got in enumerate(rp.utterances()):
                _assert_same(got, want[u], f"{hz} resident run {run} utt {u}")
        # the pre-stretch buffer stays at the native rate
        st = [u for u in range(n) if plan.speed[u] != 1.0 and abs(plan.speed[u] - 1.0) >= 0.01]
        _, _, pre = H.Oracle(small_db).synth(prm, plan.utt_ops(st[0]), float(plan.speed[st[0]]), want_pre=True)
        _assert_same(rp.read_pre(st[0], len(pre) + 64), pre, f"{hz} pre-stretch buffer")
        rp.close()
        # a session fed in pieces (an empty one among them)
        cuts = [0, 1, 9, 9, 30, 31, 50, 64]
        pieces = [plan.select(range(a, b)) for a, b in zip(cuts[:-1], cuts[1:])]
        buf = np.zeros(cap + 64, np.int16)
        soff, scnt = g.synth_pieces(pieces, prm, buf)
        for u in range(n):
            _assert_same(buf[int(soff[u]):int(soff[u]) + int(scnt[u])], want[u], f"{hz} session utt {u}")
        # texts -> PCM, in a buffer of capacity_hint at the rate
        batch = pipe.TextBatch(texts, speeds)
        tbuf = np.zeros(pipe.capacity_hint(front_small, batch, hz), np.int16)
        assert tbuf.size >= -(-pipe.capacity_hint(front_small, batch) * L // M)
        toff, tcnt, tused, _ = pipe.synth_texts(front_small, g, batch, tbuf)
        assert tused <= tbuf.size
        for u in range(n):
            _assert_same(tbuf[int(toff[u]):int(toff[u]) + int(tcnt[u])], want[u], f"{hz} synth_texts utt {u}")
    finally:
        g.close()
    # one batch over three contexts on one GPU
    ctxs = [_ctx(gpu, small_db, hz) for _ in range(3)]
    try:
        mpcm, moff, mcnt, shard = gpu.multi_synth_batch(ctxs, plan, prm)
        assert len(set(shard.tolist())) == 3
        for u in range(n):
            _assert_same(mpcm[int(moff[u]):int(moff[u]) + int(mcnt[u])], want[u], f"{hz} multi utt {u}")
    finally:
        for c in ctxs:
            c.close()


EDGE = ("tiny_stretch", "amplitude_rms0", "amplitude_rms3000", "short_units")


@pytest.mark.parametrize("hz", (8000, 16000, 48000))
@pytest.mark.parametrize("name", EDGE)
def test_edge_voices(gpu, name, hz):
    """Pre-stretch lengths 0-769 and all-zero utterances, full-scale and gain-clamped units, very short units."""
    fam = E.family(name)
    plan, prm = fam.plan(), fam.prm()
    want = [R.resample(x, hz) for x in fam.expected()]
    g = _ctx(gpu, fam.db, hz)
    try:
        rp = g.create_plan(plan, prm)
        for run in range(2):
            rp.run()
            for u, got in enumerate(rp.utterances()):
                _assert_same(got, want[u], f"{name} {hz} resident run {run} utt {u}")
        outs = g.synth_list(plan, prm)
        for u in range(plan.n_utts):
            _assert_same(outs[u], want[u], f"{name} {hz} synth_batch utt {u}")
    finally:
        g.close()


def test_native_rate_is_unchanged(gpu, small_db, batch64):
    _, _, plan, prm, native = batch64
    results = []
    for rates in ((), (22050,), (16000, 22050), (48000, 8000, 22050)):
        g = gpu.GpuSynth(small_db, 0)
        try:
            for hz in rates:
                g.set_output_rate(hz)
            rp = g.create_plan(plan, prm)
            rp.run()
            info = rp.info()
            # (slot tails past the counts are unspecified: compare the utterances)
            results.append((b"".join(x.tobytes() for x in rp.utterances()), rp.counts().tobytes(), rp.out_offsets().tobytes(),
                            info.kernel_launches, info.bound_samples, g.bounds(plan).tobytes()))
            outs = g.synth_list(plan, prm)
            for u in range(plan.n_utts):
                _assert_same(outs[u], native[u], f"rates {rates} utt {u}")
        finally:
            g.close()
    assert all(r == results[0] for r in results[1:])
    # and a converting plan enqueues exactly one more kernel (one resample launch)
    g = _ctx(gpu, small_db, 16000)
    try:
        assert g.create_plan(plan, prm).info().kernel_launches == results[0][3] + 1
    finally:
        g.close()


def test_bounds_capacity_and_short_buffers(gpu, small_db, batch64):
    _, _, plan, prm, native = batch64
    g = _ctx(gpu, small_db, 16000)
    try:
        L, M = R.ratio(16000)
        g.set_output_rate(22050)
        nb = g.bounds(plan).astype(np.int64)
        g.set_output_rate(16000)
        b = g.bounds(plan).astype(np.int64)
        assert np.array_equal(b, -(-nb * L // M))
        # a caller slot one 8-sample step short of its bound
        off = g.layout(plan).astype(np.int64)
        u = int(np.argmax(b))
        sizes = np.diff(off)
        sizes[u] = _up8(b[u]) - 8
        short = np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
        with pytest.raises(gpu.GpuError, match="-101"):
            g.synth_batch(plan, prm, out_offsets=short)
        with pytest.raises(gpu.GpuError, match="-101"):
            g.create_plan(plan, prm, short)
        # packed: the space the counts take is enough, 8 samples less is not
        _, cnt, used = g.synth_batch_packed(plan, prm, np.zeros(int(_up8(b).sum()), np.int16))
        assert used == int(_up8(cnt).sum())
        with pytest.raises(gpu.GpuError, match="-101"):
            g.synth_batch_packed(plan, prm, np.zeros(used - 8, np.int16))
        # the context is usable afterwards
        outs = g.synth_list(plan, prm)
        _assert_same(outs[5], R.resample(native[5], 16000), "after errors")
    finally:
        g.close()


def test_invalid_rates_sessions_and_mixed_multi(gpu, small_db, batch64):
    _, _, plan, prm, native = batch64
    lib = gpu.lib()
    g = gpu.GpuSynth(small_db, 0)
    try:
        for hz in (0, 7999, 48001, 96000, 44099, 47999):
            assert lib.ctts_gpu_set_output_rate(g._h, hz) == ERR_INVALID_ARG, hz
        # rejected rates leave the context at its rate
        assert np.array_equal(g.synth_list(plan, prm)[3], native[3])
        g.set_output_rate(24000)
        assert lib.ctts_gpu_set_output_rate(g._h, 8000 - 1) == ERR_INVALID_ARG
        _assert_same(g.synth_list(plan, prm)[3], R.resample(native[3], 24000), "after a rejected rate")
        # no change while a session is open
        import ctypes as C
        h = C.c_void_p()
        buf = np.zeros(1 << 20, np.int16)
        g._check(lib.ctts_gpu_session_begin(g._h, C.byref(prm), buf.ctypes.data, buf.size, None, None, C.byref(h)))
        assert lib.ctts_gpu_set_output_rate(g._h, 16000) == ERR_INVALID_ARG
        assert lib.ctts_gpu_set_output_rate(g._h, 24000) == ERR_INVALID_ARG
        assert lib.ctts_gpu_session_end(h, None) == 0
        _assert_same(g.synth_list(plan, prm)[3], R.resample(native[3], 24000), "after the session")
        # contexts of different rates do not form one multi-device batch
        g2 = gpu.GpuSynth(small_db, 0)
        try:
            with pytest.raises(gpu.GpuError, match="ctts_gpu error -1:"):
                gpu.multi_synth_batch([g, g2], plan, prm)
            g2.set_output_rate(24000)
            mpcm, moff, mcnt, _ = gpu.multi_synth_batch([g, g2], plan, prm)
            _assert_same(mpcm[int(moff[3]):int(moff[3]) + int(mcnt[3])], R.resample(native[3], 24000), "multi")
        finally:
            g2.close()
    finally:
        g.close()


def test_plan_keeps_its_rate(gpu, small_db, batch64):
    _, _, plan, prm, native = batch64
    g = _ctx(gpu, small_db, 16000)
    try:
        rp = g.create_plan(plan, prm)
        g.set_output_rate(48000)
        rp.run()
        got = rp.utterances()
        for u in (0, 10, 63):
            _assert_same(got[u], R.resample(native[u], 16000), f"plan of 16 kHz utt {u}")
        _assert_same(g.synth_list(plan, prm)[10], R.resample(native[10], 48000), "context at 48 kHz")
    finally:
        g.close()


def test_full_batch_at_16k(H, gpu):
    """BASELINE configs[2] (4096 utterances) at 16 kHz: every count is ceil(native * L / M) of the 22 050 Hz run,
    and 64 utterances equal the oracle."""
    db = H.synthetic_db()
    fr = H.front.Front(db, H.shipped_config(), H.NORM_CSV)
    prm = fr.params()
    plan = fr.plan(H.corpus.batch(4096, seed=1234))
    g = gpu.GpuSynth(db, 0)
    try:
        rp = g.create_plan(plan, prm)
        rp.run()
        native_cnt = rp.counts().astype(np.int64)
        rp.close()
        g.set_output_rate(16000)
        L, M = R.ratio(16000)
        rp = g.create_plan(plan, prm)
        rp.run()
        cnt = rp.counts().astype(np.int64)
        assert np.array_equal(cnt, -(-native_cnt * L // M))
        assert (cnt <= g.bounds(plan).astype(np.int64)).all()
        off = rp.out_offsets().astype(np.int64)
        orc = H.Oracle(db)
        pick = sorted(np.random.default_rng(5).choice(4096, 64, replace=False).tolist())
        for u in pick:
            want = R.resample(orc.synth(prm, plan.utt_ops(u), 1.0)[0], 16000)
            _assert_same(rp.read_pcm(int(off[u]), int(cnt[u])), want, f"utt {u}")
    finally:
        g.close()


def test_command_line_writes_the_rate(H, golden, small_db, tmp_path):
    b = H.importlib.import_module("2026-simple-c-tts_b200._build")
    exe = b.build_cli()
    shutil.copy(H.SHIPPED_YAML, tmp_path / "config.yaml")
    shutil.copy(H.NORM_CSV, tmp_path / "normalization.csv")
    (tmp_path / "voice.db").write_bytes(small_db)
    for k, speed in enumerate(("1.0", "1.5")):
        for hz in (16000, 44100):
            r = subprocess.run([exe, "synth", "voice.db", "olá mundo", f"o{k}_{hz}.wav", speed, str(hz)], cwd=tmp_path,
                               capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            raw = (tmp_path / f"o{k}_{hz}.wav").read_bytes()
            want = R.resample(golden[f"e2e_pcm_{k}"], hz)
            assert len(raw) == 44 + 2 * len(want)
            assert struct.unpack("<IHHIIHH", raw[16:36]) == (16, 1, 1, hz, 2 * hz, 2, 16)
            assert struct.unpack("<I", raw[40:44])[0] == 2 * len(want)
            assert np.array_equal(np.frombuffer(raw[44:], dtype="<i2"), want)
    (tmp_path / "t.tsv").write_text("1.0\tolá mundo\n1.5\tolá mundo\n", encoding="utf-8")
    r = subprocess.run([exe, "synth-batch", "voice.db", "t.tsv", "out", "16000"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "out" / "000000.wav").read_bytes() == (tmp_path / "o0_16000.wav").read_bytes()
    assert (tmp_path / "out" / "000001.wav").read_bytes() == (tmp_path / "o1_16000.wav").read_bytes()
    r = subprocess.run([exe, "synth", "voice.db", "olá mundo", "bad.wav", "1.0", "44099"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and not (tmp_path / "bad.wav").exists()
