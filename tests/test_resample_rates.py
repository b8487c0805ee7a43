"""CPU tests of the output-rate conversion over the whole accepted rate space (DESIGN.md 3.4).

test_resample.py checks the filter and the oracle at the common rates.  Here:
  * the accepted set, every integer from 7 000 to 50 000;
  * the launch geometry of resample_kernel (ctts_host_resample_geometry) against the kernel's tile arithmetic,
    restated in integer numpy from resample.cuh, for all 4 593 accepted rates: the staging bound, every tap read,
    the tile count, and the 48 KB of shared memory every rate stays under;
  * taps, response and the ±1 LSB agreement with scipy at a stratified set of extreme rates (RATES below).
"""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

import resample_oracle as R
from test_resample import _inputs, _resample_poly_int16, _scipy_taps, _ulps

scipy_signal = pytest.importorskip("scipy.signal")

RS_THREADS, RS_COPIES = 256, 4   # resample.cuh
SMEM_DEFAULT = 48 * 1024         # dynamic shared memory a kernel gets without cudaFuncSetAttribute

# Rates that sit at the ends of what changes with the rate: L (phases; L > RS_THREADS spreads one row of items
# over several tiles), M/L, the tap count N = 80 max(L, M) + 1, the staging per tile, and how many rows of
# RS_COPIES * L outputs one tile spans.
RATES = {
    8000: "160/441: the largest M/L, kp = 224",
    8015: "229/630: the largest staging of any accepted rate",
    8785: "251/630: L just below 256, a tile spans 3 rows",
    8995: "257/630: L just above 256, a tile spans 2 rows and a row spreads over 2 tiles",
    10752: "256/525: L = RS_THREADS exactly",
    12800: "256/441: L = RS_THREADS, the largest M of the L = 256 rates",
    8820: "2/5: many rows per tile",
    9450: "3/7: many rows per tile",
    11025: "1/2: L = 1",
    14700: "2/3: many rows per tile",
    33075: "3/2: many rows per tile, upsampling",
    22025: "881/882: ratio just below 1 with a large L",
    22075: "883/882: ratio just above 1 with a large L",
    22400: "64/63",
    25525: "1021/882: L near the limit",
    30720: "1024/735: L = 1024, N = 81 921 taps",
    43008: "1024/525: L = 1024, N = 81 921 taps",
    46035: "1023/490",
    48000: "320/147: the smallest M/L",
}


def _gcd_rule(hz):
    g = math.gcd(hz, R.NATIVE)
    L, M = hz // g, R.NATIVE // g
    return (L, M) if 8000 <= hz <= 48000 and max(L, M) <= 1024 else None


ACCEPTED = [hz for hz in range(8000, 48001) if _gcd_rule(hz) is not None]


def test_accepted_set_is_the_gcd_rule():
    for hz in range(7000, 50001):
        assert R.ratio(hz) == _gcd_rule(hz), hz
    assert len(ACCEPTED) == 4593
    assert sum(_gcd_rule(hz)[0] > RS_THREADS for hz in ACCEPTED) == 2916


def _geometry_fn():
    lib = importlib.import_module("2026-simple-c-tts_b200.gpu").lib()
    f = lib.ctts_host_resample_geometry
    u32p = C.POINTER(C.c_uint32)
    f.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, u32p, u32p, u32p, u32p]
    f.restype = None
    return f


def geometry(L, M, max_out=0, fn=None):
    """(kp, c, smem_floats, tiles) as libctts_gpu.so computes them."""
    v = [C.c_uint32() for _ in range(4)]
    (fn or _geometry_fn())(L, M, max_out, *[C.byref(x) for x in v])
    return tuple(int(x.value) for x in v)


# ---------------------------------------------------------------------------------- resample_kernel, restated

def _first_out(w, L):
    return (w // L) * (L * RS_COPIES) + w % L


def tile_model(L, M, kp, c, w0, n_out, threads=True):
    """resample.cuh lines 45-84 for tiles starting at work items w0 of utterances of n_out outputs (int64 arrays
    of one shape).  Returns, per tile: live (the tile passes both early returns), span, and with `threads` the
    least base[0] and the largest base[q] over the tile's threads with an output (the reads of a thread are
    base[q] .. base[q] + kp - 1)."""
    row = L * RS_COPIES
    items = -(-n_out // row) * L
    w_last = np.minimum(items, w0 + RS_THREADS) - 1
    m_first = _first_out(w0, L)
    live = (w0 < items) & (m_first < n_out)
    m_last = np.minimum(n_out - 1, _first_out(w_last, L) + (RS_COPIES - 1) * L)
    x_lo = (m_first * M + c) // L - kp + 1
    x_hi = (m_last * M + c) // L
    span = x_hi - x_lo + 1
    if not threads:
        return live, span, None, None
    w = w0[:, None] + np.arange(RS_THREADS)
    m0 = _first_out(w, L)
    th = live[:, None] & (w <= w_last[:, None]) & (m0 < n_out[:, None])
    jmax0 = (m0 * M + c) // L
    base0 = jmax0 - kp + 1 - x_lo[:, None]
    # base[q] grows with q (jm = jmax0 + q M): the last live q gives a thread's largest read
    q_last = np.minimum((n_out[:, None] - 1 - m0) // L, RS_COPIES - 1)
    base_last = base0 + np.where(th, q_last, 0) * M
    lo = np.where(th, base0, np.iinfo(np.int64).max).min(axis=1)
    hi = np.where(th, base_last, np.iinfo(np.int64).min).max(axis=1)
    return live, span, lo, hi


def _check_tiles(hz, L, M, kp, smem_floats, live, span, lo, hi):
    assert (span[live] >= 1).all(), hz
    assert span[live].max(initial=0) <= smem_floats, (hz, int(span[live].max()), smem_floats)
    if lo is not None:
        assert (lo[live] >= 0).all(), hz
        assert (hi[live] + kp - 1 < span[live]).all(), hz


def test_staging_bound_every_rate():
    """Every accepted rate, every tile class (w0 = 256 b, b < L: the pattern of spans repeats with period L),
    unclipped: the span fits the host's bound, every tap read of every thread lies inside the span."""
    fn = _geometry_fn()
    worst, margin = (0, None), []
    for hz in ACCEPTED:
        L, M = _gcd_rule(hz)
        kp, c, smem_floats, _ = geometry(L, M, 0, fn)
        assert kp % 4 == 0 and kp * L >= 80 * max(L, M) + 1 and c == 40 * max(L, M)
        assert smem_floats % 4 == 0
        w0 = np.arange(L, dtype=np.int64) * RS_THREADS
        live, span, lo, hi = tile_model(L, M, kp, c, w0, np.full(L, 1 << 40, np.int64))
        assert live.all()
        _check_tiles(hz, L, M, kp, smem_floats, live, span, lo, hi)
        worst = max(worst, (smem_floats * 4, hz))
        if hz != R.NATIVE:
            margin.append((smem_floats - int(span.max()), hz))
    # no accepted rate needs more than the default 48 KB: set_output_rate's cudaFuncSetAttribute branch is dead
    assert worst[0] <= SMEM_DEFAULT and worst[1] == 8015, worst
    # the bound is 6 floats above the largest span at 11 025 and 33 075 Hz, more elsewhere: a change to it shows here
    assert sorted(margin)[:2] == [(6, 11025), (6, 33075)], sorted(margin)[:4]


def _clipped_cases(L, n_rows):
    """(w0, n_out) of the tiles that hold the last row of an utterance ending in that row: for the first n_rows
    row indices r (so the last row starts at every residue of r L mod 256 they reach), n_out = r row + k for k at
    the ends of the row's four copies."""
    row = L * RS_COPIES
    w0s, nos = [], []
    for r in range(n_rows):
        first, last = r * L // RS_THREADS, ((r + 1) * L - 1) // RS_THREADS + 1   # tiles touching row r (+ one past)
        for k in sorted({1, 2, L - 1, L, L + 1, 2 * L, 3 * L - 1, 3 * L, 3 * L + 1, row - 1, row} - {0}):
            b = np.arange(first, last + 1, dtype=np.int64)
            w0s.append(b * RS_THREADS)
            nos.append(np.full(len(b), r * row + k, np.int64))
    return np.concatenate(w0s), np.concatenate(nos)


def test_staging_bound_clipped_last_tiles():
    """Every accepted rate, last tiles clipped by n_out at the ends of a row, the last row at every tile alignment
    its first rows reach (tile level).  Some of these tiles hold only past-the-end items (a tile that starts inside
    the last row after its last live item) and return before staging."""
    fn = _geometry_fn()
    empty_seen = 0
    for hz in ACCEPTED:
        L, M = _gcd_rule(hz)
        kp, c, smem_floats, _ = geometry(L, M, 0, fn)
        n_rows = min(RS_THREADS // math.gcd(L, RS_THREADS) + 1, 64)
        w0, n_out = _clipped_cases(L, n_rows)
        live, span, _, _ = tile_model(L, M, kp, c, w0, n_out, threads=False)
        _check_tiles(hz, L, M, kp, smem_floats, live, span, None, None)
        items = -(-n_out // (L * RS_COPIES)) * L
        empty_seen += int(((w0 < items) & ~live).sum())
    assert empty_seen > 0


@pytest.mark.parametrize("hz", sorted(RATES))
def test_tiles_at_the_stratified_rates(hz):
    """Per thread, for clipped last tiles; and the whole grid of tiles() tiles for utterances of many lengths
    produces every output exactly once."""
    L, M = R.ratio(hz)
    kp, c, smem_floats, _ = geometry(L, M)
    w0, n_out = _clipped_cases(L, min(RS_THREADS // math.gcd(L, RS_THREADS) + 1, 64))
    live, span, lo, hi = tile_model(L, M, kp, c, w0, n_out)
    _check_tiles(hz, L, M, kp, smem_floats, live, span, lo, hi)
    row = L * RS_COPIES
    for n in (1, 2, row - 1, row, row + 1, 3 * row + L, 7 * row + 2 * L - 1, 256 * row + 1):
        tiles = geometry(L, M, n)[3]
        w0 = np.arange(tiles, dtype=np.int64) * RS_THREADS
        nn = np.full(tiles, n, np.int64)
        live, span, lo, hi = tile_model(L, M, kp, c, w0, nn)
        _check_tiles(hz, L, M, kp, smem_floats, live, span, lo, hi)
        # every output m < n is written by exactly one (tile, thread, copy) of the grid
        w = (w0[:, None] + np.arange(RS_THREADS)).ravel()
        items = -(-n // row) * L
        w = w[w < items]
        m = (_first_out(w, L)[:, None] + L * np.arange(RS_COPIES)).ravel()
        m = np.sort(m[m < n])
        assert np.array_equal(m, np.arange(n)), (hz, n)
        assert (tiles - 1) * RS_THREADS < max(items, 1)   # and no more tiles than that


def test_tile_count_covers_long_utterances():
    fn = _geometry_fn()
    for hz in ACCEPTED[::7] + sorted(RATES):
        L, M = _gcd_rule(hz)
        row = L * RS_COPIES
        for n in (0, 1, row, row + 1, 1 << 31, 0xffffffff - 16):
            tiles = geometry(L, M, n, fn)[3]
            items = -(-n // row) * L
            assert tiles >= 1 and tiles * RS_THREADS >= items and (tiles - 1) * RS_THREADS < max(items, 1), (hz, n)


# ---------------------------------------------------------------------------------- filter at the extreme rates

@pytest.mark.parametrize("hz", sorted(RATES))
def test_taps_at_the_stratified_rates(hz):
    L, M = R.ratio(hz)
    g = R.taps(hz)
    assert len(g) == 80 * max(L, M) + 1
    assert _ulps(g, _scipy_taps(hz).astype(np.float32)).max() <= 1
    lib = importlib.import_module("2026-simple-c-tts_b200.gpu").lib()
    lib.ctts_host_resample_taps.argtypes = [C.c_uint, C.c_uint, C.c_void_p]
    lib.ctts_host_resample_taps.restype = None
    p = np.zeros_like(g)
    lib.ctts_host_resample_taps(L, M, p.ctypes.data)
    assert _ulps(p, g).max() <= 1


@pytest.mark.parametrize("hz", sorted(RATES))
def test_response_at_the_stratified_rates(hz):
    """DESIGN.md 3.4: passband ripple <= 0.0033 dB up to 0.44 f_low; rejection from 0.5 f_low on >= 69.4 dB at
    R = 2, >= 69.5 dB for R <= 37 and >= 70.0 dB above.  Evaluated on an FFT grid at least 32 times denser than the
    filter is long."""
    L, M = R.ratio(hz)
    g = R.taps(hz).astype(np.float64) / L
    f_low = min(R.NATIVE, hz)
    fs = R.NATIVE * L
    nfft = 1 << max(20, int(math.ceil(math.log2(32 * len(g)))))
    h = np.abs(np.fft.rfft(g, nfft))
    f = np.arange(len(h)) * fs / nfft
    ripple = 20 * np.log10(h[f <= 0.44 * f_low])
    assert np.abs(ripple).max() <= 0.0033, ripple.max()
    R_ = max(L, M)
    assert 20 * np.log10(h[f >= 0.5 * f_low].max()) <= (-69.4 if R_ <= 2 else -69.5 if R_ <= 37 else -70.0)


@pytest.mark.parametrize("hz", sorted(RATES))
def test_oracle_within_one_lsb_of_scipy_at_the_stratified_rates(hz):
    rng = np.random.default_rng(hz)
    for x in _inputs(rng):
        y = R.resample(x, hz)
        z = _resample_poly_int16(x, hz)
        assert len(y) == len(z) == R.count(hz, len(x))
        assert np.abs(y.astype(np.int64) - z).max() <= 1
