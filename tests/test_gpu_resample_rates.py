"""GPU tests of the output-rate conversion across the accepted rate space and at the launch limits
(ctts_gpu_set_output_rate, resample_kernel; DESIGN.md 3.4).

  * every integer rate in [7 990, 48 010]: accepted by the device exactly when the oracle accepts it, with a table;
  * at the stratified rates of test_resample_rates.RATES, constructed voices whose output lengths put the last
    tile of an utterance on every edge of the kernel's geometry, bit for bit against the oracle;
  * more than 65 535 utterances in one launch (grid.y is split in chunks: resample, WSOLA verify, pack copy);
  * more than 2^32 output samples in one plan (configs[2] at 48 kHz).

Run on a B200 with:  python -m pytest tests/test_gpu_resample_rates.py -m gpu
"""
import math

import numpy as np
import pytest

import edge_voices as E
import resample_oracle as R
from test_gpu_resample import _assert_same, _up8
from test_resample_rates import RATES, RS_COPIES, RS_THREADS, _first_out

GRID_Y = 65535


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


def _ctx(gpu, db, hz):
    g = gpu.GpuSynth(db, 0)
    g.set_output_rate(hz)
    return g


def _read_all(rp):
    """Every utterance of a resident plan, from one read of its whole buffer."""
    cnt = rp.counts().astype(np.int64)
    off = rp.out_offsets().astype(np.int64)
    pcm = rp.read_pcm(0, int(off[-1]))
    return cnt, off, pcm


# ---------------------------------------------------------------------------------- acceptance on the device

@pytest.mark.gpu
def test_device_accepts_exactly_the_oracles_rates(gpu, small_db):
    lib = gpu.lib()
    g, built = None, 0
    try:
        for hz in range(7990, 48011):
            if g is None or built >= 300:   # contexts keep every table they build: bound the device memory
                if g is not None:
                    g.close()
                g, built = gpu.GpuSynth(small_db, 0), 0
            rc = lib.ctts_gpu_set_output_rate(g._h, hz)
            assert (rc == 0) == (R.ratio(hz) is not None), (hz, rc)
            built += rc == 0
    finally:
        if g is not None:
            g.close()


# ---------------------------------------------------------------------------------- tile edges

def _n_for(hz, t):
    """The least native length whose output has at least t samples."""
    L, M = R.ratio(hz)
    return 0 if t <= 0 else (t - 1) * M // L + 1


def _empty_tile(L, n_out):
    """Whether the utterance's last tile with items holds only past-the-end items (resample.cuh: m_first >= n_out)."""
    row = L * RS_COPIES
    items = -(-n_out // row) * L
    b = np.arange(-(-items // RS_THREADS), dtype=np.int64)
    return bool((_first_out(b * RS_THREADS, L) >= n_out).any())


def edge_classes(hz, n_out):
    """The geometry classes an output length reaches at hz."""
    L, M = R.ratio(hz)
    row, s = L * RS_COPIES, -(-L // M)   # s: the least step of n_out between native lengths
    items = -(-n_out // row) * L
    g = math.gcd(L, RS_THREADS)
    cls = set()
    if n_out == 0:
        cls.add("zero")
    if 1 <= n_out <= s:
        cls.add("first")
    if n_out == 2 and s == 1:
        cls.add("two")
    if n_out > row:
        r = n_out % row
        if r == 0:
            cls.add("row_end")
        elif r <= s:
            cls.add("above_row")
        elif r >= row - s:
            cls.add("below_row")
    if g < RS_THREADS and items > RS_THREADS and items % RS_THREADS == g:
        cls.add("items_above_256")
    if n_out and _empty_tile(L, n_out):
        cls.add("empty_tile")
    return cls


def targeted(hz):
    """The classes the construction aims at for hz (those the rate can reach)."""
    L, M = R.ratio(hz)
    want = {"zero", "first", "row_end", "above_row", "below_row"}
    if L <= M:
        want.add("two")
    if math.gcd(L, RS_THREADS) < RS_THREADS:
        want.add("items_above_256")
    if L > RS_THREADS or _empty_row(L, M) is not None:
        want.add("empty_tile")
    return want


def _empty_row(L, M):
    """A row index r such that an utterance ending just past the start of row r leaves a tile of dead items."""
    s = -(-L // M)
    for r in range(1, 2 * RS_THREADS + 1):
        lo, hi = r * L + s, r * L + L - 1   # a tile starting in [lo, hi] has no live item
        if hi >= lo and (hi // RS_THREADS) * RS_THREADS >= lo:
            return r
    return None


def edge_lengths(hz):
    """Native lengths whose outputs at hz hit the targeted classes."""
    L, M = R.ratio(hz)
    row = L * RS_COPIES
    outs = {0, 1, 2} | {k * row + d for k in (1, 2, 3) for d in (-1, 0, 1)}
    # (upsampling skips output lengths) 4 k M native samples give exactly k rows of outputs; one sample less or more ends just below or above a row
    native = {d + 4 * k * M for k in (1, 2, 3) for d in (-1, 0, 1)}
    g = math.gcd(L, RS_THREADS)
    if g < RS_THREADS:
        # rows * L = g (mod 256): the last tile holds g items
        rows = next(r for r in range(1, 2 * RS_THREADS + 2) if r * L % RS_THREADS == g and r * L > RS_THREADS)
        outs |= {(rows - 1) * row + 1, rows * row}
    r = _empty_row(L, M)
    if r is not None:
        outs.add(r * row + 1)
    return sorted(native | {_n_for(hz, t) for t in outs})


def family_rate_edges(hz, seed=21):
    """Single-unit utterances at speed 1.0 with no pause, fades, trim or crossfade: an utterance's native length
    is its unit's length, chosen by edge_lengths."""
    rng = np.random.default_rng(seed + hz)
    cfg = E.H.shipped_config()
    cfg.word_pause_ms = 0.0
    cfg.fade_in_ms = 0.0
    cfg.fade_out_ms = 0.0
    cfg.remove_word_silence = 0
    cfg.crossfade_ms = 0.0
    names = E.Names()
    units, words = [], []
    for n in edge_lengths(hz):
        nm = names.take("other")
        units.append((nm, E.harmonic(rng, n)))
        words.append([[nm]])
    return E.Family(f"rate_edges_{hz}", units, words, [1.0] * len(words), cfg, params={"fade_in_samples": 0})


_families = {}


def rate_family(hz):
    if hz not in _families:
        _families[hz] = family_rate_edges(hz)
    return _families[hz]


@pytest.mark.parametrize("hz", sorted(RATES))
def test_rate_edge_witness(hz):
    """CPU: from the oracle's native lengths, every targeted class is reached at hz."""
    fam = rate_family(hz)
    native = fam.expected()
    assert [len(x) for x in native] == edge_lengths(hz)
    seen = set().union(*(edge_classes(hz, R.count(hz, len(x))) for x in native))
    assert targeted(hz) <= seen, (hz, targeted(hz) - seen)


def _parity(gpu, fam, hz, what):
    plan, prm = fam.plan(), fam.prm()
    want = [R.resample(x, hz) for x in fam.expected()]
    g = _ctx(gpu, fam.db, hz)
    try:
        rp = g.create_plan(plan, prm)
        for run in range(2):
            rp.run()
            cnt, off, pcm = _read_all(rp)
            for u in range(plan.n_utts):
                _assert_same(pcm[off[u]:off[u] + cnt[u]], want[u], f"{what} {hz} resident run {run} utt {u}")
        outs = g.synth_list(plan, prm)
        for u in range(plan.n_utts):
            _assert_same(outs[u], want[u], f"{what} {hz} synth_batch utt {u}")
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("hz", sorted(RATES))
def test_rate_edges_match_the_oracle(gpu, hz):
    _parity(gpu, rate_family(hz), hz, "rate edges")


@pytest.mark.gpu
@pytest.mark.parametrize("hz", sorted(RATES))
@pytest.mark.parametrize("name", ("amplitude_rms3000", "tiny_stretch"))
def test_edge_families_at_the_stratified_rates(gpu, name, hz):
    """Saturation (full-scale units) and zero-length and one-sample utterances at every stratified rate."""
    _parity(gpu, E.family(name), hz, name)


# ---------------------------------------------------------------------------------- more than 65 535 utterances

PAIRS = [("olá", 1.5), ("bom dia", 0.75), ("casa", 1.25), ("sim", 0.6180339), ("não", 2.0), ("mar azul", 1.2345678),
         ("olá dia", 1.0)]
N_BIG = 80000


@pytest.fixture(scope="module")
def big_batch(front_small, oracle_small):
    """N_BIG short utterances from a few (text, speed) pairs, the oracle's PCM once per pair.  Utterance u uses
    pair u % 7 (7 does not divide 65 535, so the two grid.y chunks hold different pairs at the same index); 6 in
    7 are stretched, more than 65 535 of them."""
    pick = np.arange(N_BIG) % len(PAIRS)
    texts = [PAIRS[k][0] for k in pick]
    speeds = [PAIRS[k][1] for k in pick]
    plan = front_small.plan(texts, speeds)
    prm = front_small.params()
    first = {int(k): int(np.argmax(pick == k)) for k in np.unique(pick)}
    native = {k: oracle_small.synth(prm, plan.utt_ops(u), float(speeds[u]))[0] for k, u in first.items()}
    assert sum(PAIRS[k][1] != 1.0 for k in pick) > GRID_Y
    return plan, prm, pick, native


def _check_big(cnt, off, pcm, pick, want, what):
    want_cnt = np.array([len(want[k]) for k in range(len(PAIRS))], np.int64)[pick]
    bad = np.nonzero(cnt != want_cnt)[0]
    assert not len(bad), f"{what}: {len(bad)} counts differ, first at {bad[:5]}"
    for u in range(len(pick)):
        _assert_same(pcm[off[u]:off[u] + cnt[u]], want[pick[u]], f"{what} utt {u}")


@pytest.mark.gpu
def test_more_than_65535_utterances(gpu, small_db, big_batch, monkeypatch):
    monkeypatch.setenv("CTTS_GPU_CHUNK_SAMPLES", str(1 << 40))   # read at init: one chunk holds the whole batch
    plan, prm, pick, native = big_batch
    # native rate: the WSOLA verify launch is split without the resampler
    g = gpu.GpuSynth(small_db, 0)
    try:
        rp = g.create_plan(plan, prm)
        info = rp.info()
        assert info.n_stretch > GRID_Y
        launches_native = info.kernel_launches
        rp.run()
        _check_big(*_read_all(rp), pick, native, "22050 Hz resident")
        rp.close()
        # 16 kHz: two resample launches on top of the same kernels
        hz = 16000
        g.set_output_rate(hz)
        want = {k: R.resample(x, hz) for k, x in native.items()}
        rp = g.create_plan(plan, prm)
        assert rp.info().n_stretch > GRID_Y
        assert rp.info().kernel_launches == launches_native + 2
        for run in range(2):
            rp.run()
            _check_big(*_read_all(rp), pick, want, f"{hz} resident run {run}")
        rp.close()
        # a session of one piece of every utterance: two pack copy launches
        cap = int(_up8(g.bounds(plan).astype(np.int64)).sum()) + 64
        buf = np.zeros(cap, np.int16)
        soff, scnt = g.synth_pieces([plan], prm, buf)
        _check_big(scnt.astype(np.int64), soff.astype(np.int64), buf, pick, want, f"{hz} session")
    finally:
        g.close()


# ---------------------------------------------------------------------------------- more than 2^32 output samples

def _mem_available():
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


@pytest.mark.gpu
def test_more_than_2_to_32_output_samples(H, gpu):
    """BASELINE configs[2] (4096 utterances) at 48 kHz: more than 2^32 output samples.  Every count is
    ceil(native * L / M) of the 22 050 Hz run; 64 utterances equal the oracle, the last 16 by offset among them,
    all of which start above 2^32."""
    db = H.synthetic_db()
    fr = H.front.Front(db, H.shipped_config(), H.NORM_CSV)
    prm = fr.params()
    plan = fr.plan(H.corpus.batch(4096, seed=1234))
    hz = 48000
    L, M = R.ratio(hz)
    g = gpu.GpuSynth(db, 0)
    try:
        rp = g.create_plan(plan, prm)
        rp.run()
        native_cnt = rp.counts().astype(np.int64)
        rp.close()
        g.set_output_rate(hz)
        rp = g.create_plan(plan, prm)
        assert rp.out_samples > 1 << 32
        rp.run()
        cnt = rp.counts().astype(np.int64)
        assert np.array_equal(cnt, -(-native_cnt * L // M))
        off = rp.out_offsets().astype(np.int64)
        last = np.argsort(off[:-1])[-16:]
        assert (off[last] > 1 << 32).all()
        pick = sorted(set(np.random.default_rng(6).choice(4096, 48, replace=False).tolist()) | set(last.tolist()))
        orc = H.Oracle(db)
        want = {u: R.resample(orc.synth(prm, plan.utt_ops(u), 1.0)[0], hz) for u in pick}
        for u in pick:
            _assert_same(rp.read_pcm(int(off[u]), int(cnt[u])), want[u], f"resident utt {u}")
        rp.close()
        # the packed layout into a host buffer of more than 2^32 samples
        cap = int(_up8(g.bounds(plan).astype(np.int64)).sum())
        assert cap > 1 << 32
        need = 2 * cap + (8 << 30)
        if _mem_available() < need:
            pytest.skip(f"synth_batch_packed into {2 * cap >> 30} GiB of host memory: "
                        f"{_mem_available() >> 30} GiB available, {need >> 30} GiB wanted")
        buf = np.zeros(cap, np.int16)
        poff, pcnt, used = g.synth_batch_packed(plan, prm, buf)
        assert np.array_equal(pcnt.astype(np.int64), cnt)
        assert used > 1 << 32 and (poff.astype(np.int64)[last] > 1 << 32).all()
        for u in pick:
            _assert_same(buf[int(poff[u]):int(poff[u]) + int(pcnt[u])], want[u], f"packed utt {u}")
    finally:
        g.close()
