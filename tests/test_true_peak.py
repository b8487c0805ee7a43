"""CPU tests of the true-peak ceiling of the loudness normalization (ctts_gpu_set_loudness_true_peak, DESIGN.md 3.6
and 5): the product's interpolator taps equal the formula; the oracle's true peak P (tests/true_peak_oracle.c) equals
a float64 numpy restatement, a full convolution of the 4x zero-stuffed signal with the float taps; and over thousands
of seeded signals the guarantee holds: the interpolated peak of the delivered y, in float64, is at most A."""
import ctypes as C
import importlib

import numpy as np
import pytest

import loudness_oracle as O
import true_peak_oracle as TP

SQUARE4_DB = 3.11   # the period-4 full-scale square over its sample peak, on this interpolator


def formula_taps() -> np.ndarray:
    """The contract's taps, restated in numpy: float64, |h| <= 1e-9 to 0, rounded to float32 once."""
    j = np.arange(49, dtype=np.float64)
    h = np.sinc((j - 24.0) / 4.0) * 0.5 * (1.0 - np.cos(2.0 * np.pi * j / 48.0))
    h[np.abs(h) <= 1e-9] = 0.0
    return h.astype(np.float32)


def interpolated(x: np.ndarray, h: np.ndarray | None = None) -> np.ndarray:
    """v[m], m = -24 .. 4(n - 1) + 24, in float64: the 4x zero-stuffed x convolved with the float taps."""
    h = formula_taps() if h is None else h
    x = np.asarray(x, np.float64)
    if len(x) == 0:
        return np.zeros(0)
    s = np.zeros(4 * len(x) - 3)
    s[::4] = x
    return np.convolve(s, h.astype(np.float64))


def peak64(x) -> float:
    v = interpolated(x)
    return float(np.abs(v).max()) if len(v) else 0.0


def square4(n: int, amp: int = 32767) -> np.ndarray:
    """The period-4 square amp, amp, -amp, -amp, ..."""
    return np.where(np.arange(n) % 4 < 2, amp, -amp).astype(np.int16)


def test_product_taps_equal_the_formula():
    lib = importlib.import_module("2026-simple-c-tts_b200.gpu").lib()
    lib.ctts_host_true_peak_taps.argtypes = [C.c_void_p]
    lib.ctts_host_true_peak_taps.restype = None
    got = np.zeros(49, np.float32)
    lib.ctts_host_true_peak_taps(got.ctypes.data)
    want = formula_taps()
    assert got.tobytes() == want.tobytes()
    assert TP.taps().tobytes() == want.tobytes()
    # phase 0 is the identity
    assert got[24] == 1.0 and np.count_nonzero(got[0::4]) == 1
    h = got.astype(np.float64)
    dc = [h[r::4].sum() for r in (1, 2, 3)]
    l1 = [np.abs(h[r::4]).sum() for r in (1, 2, 3)]
    assert [len(h[r::4]) for r in (1, 2, 3)] == [12, 12, 12]
    assert np.allclose(dc, [1.00048, 1.00090, 1.00048], atol=5e-6), dc
    assert np.allclose(l1, [1.631, 1.864, 1.631], atol=5e-4), l1
    # response relative to DC at 0.1, 0.4, 0.45 fs (the interpolator's passband at the input rate)
    f = np.array([0.1, 0.4, 0.45])
    H = np.abs(np.exp(-2j * np.pi * np.outer(f / 4.0, np.arange(49))) @ h) / h.sum()
    assert np.allclose(20 * np.log10(H), [-0.004, -0.44, -2.2], atol=0.05), 20 * np.log10(H)


def _signals():
    rng = np.random.default_rng(2024)
    out = [(f"len{n}", rng.integers(-32768, 32768, n).astype(np.int16)) for n in range(61)]
    out += [(f"noise{k}", rng.integers(-32768, 32768, int(rng.integers(100, 3000))).astype(np.int16)) for k in range(10)]
    out += [(f"quiet{k}", rng.integers(-30, 31, int(rng.integers(100, 3000))).astype(np.int16)) for k in range(5)]
    out += [("full_scale", np.where(rng.random(2000) < 0.5, -32768, 32767).astype(np.int16))]
    out += [("dc", np.full(500, 32767, np.int16)), ("dc_neg", np.full(37, -32768, np.int16))]
    for n in (1, 2, 7, 100):
        for at in (0, n - 1):
            x = np.zeros(n, np.int16)
            x[at] = -32768
            out.append((f"impulse{n}_{at}", x))
    out += [("square4", square4(1000))]
    return out


@pytest.mark.parametrize("name,x", _signals(), ids=[n for n, _ in _signals()])
def test_oracle_equals_numpy(name, x):
    P = TP.true_peak(x)
    want = peak64(x)
    assert abs(P - want) <= 1e-6 * max(want, 1.0), (name, P, want)
    assert P >= (np.abs(x.astype(np.int32)).max() if len(x) else 0)
    assert np.float32(P) == P


def test_square_reads_plus_3_11_db():
    P = TP.true_peak(square4(4000))
    assert abs(20 * np.log10(P / 32767) - SQUARE4_DB) < 0.005, 20 * np.log10(P / 32767)


def guarantee_signals(seed: int = 7):
    """(fs, T, C, x) over thousands of seeded cases: noise, fs/4 and fs/2 full-scale patterns, quiet signals that the
    gain amplifies up to the table's reach, single impulses in silence, tones near Nyquist; every one long enough
    (>= 400 ms) for L to be defined."""
    rng = np.random.default_rng(seed)
    for k in range(3000):
        fs = int(rng.choice([8000, 11025, 16000]))
        n = int(rng.integers(4 * fs // 10, 4 * fs // 10 + 1500))
        kind = k % 6
        if kind == 0:
            x = rng.integers(-32768, 32768, n)
        elif kind == 1:
            x = np.roll(square4(n), int(rng.integers(0, 4))).astype(np.int64)
        elif kind == 2:
            x = np.where(np.arange(n) % 2, -32768, 32767)
        elif kind == 3:
            amp = int(rng.integers(1, 40))
            x = rng.integers(-amp, amp + 1, n)
        elif kind == 4:
            x = np.zeros(n, np.int64)
            x[int(rng.integers(0, n))] = int(rng.choice([-32768, 32767, int(rng.integers(-32768, 32768))]))
        else:
            f = rng.uniform(0.35, 0.5) * fs
            amp = float(rng.choice([32767.0, rng.uniform(1.0, 32767.0)]))
            x = np.round(amp * np.sin(2 * np.pi * f * np.arange(n) / fs + rng.uniform(0, 6.3)))
        x = np.clip(x, -32768, 32767).astype(np.int16)
        T = float(np.float32(rng.uniform(-60.0, -5.0)))
        C = float(np.float32(rng.choice([0.0, -1.0, -2.0, rng.uniform(-20.0, 0.0)])))
        yield fs, T, C, x


def test_guarantee_over_seeded_signals():
    worst, amplified, limited = -np.inf, 0, 0
    for fs, T, C, x in guarantee_signals():
        y, L, G, P = TP.normalize(x, fs, T, C)
        A = O.ceiling(C)
        if not np.isfinite(L):
            assert G == O.UNITY
            continue
        Gs = O.gain(L, T, C, int(np.abs(x.astype(np.int32)).max()))
        assert G <= Gs, (fs, T, C, G, Gs)
        margin = peak64(y) - A
        assert margin <= 0.0, (fs, T, C, G, P, margin)
        worst = max(worst, margin)
        amplified += G > 4 * O.UNITY
        limited += G < Gs
    assert amplified > 100 and limited > 300, (amplified, limited)
    assert worst < 0.0


def test_gain_rule():
    for L, T, C, P in [(-20.0, -16.0, -1.0, 30000.5), (-40.0, -16.0, -1.0, 100.25), (-16.0, -16.0, -1.0, 32767.0)]:
        A = O.ceiling(C)
        k = int(np.floor(100 * (np.float32(T) - L) + 0.5))
        want = min(int(O.table()[k + O.K_MAX]), int(np.floor((A - 1) * 65536.0 / P)))
        assert TP.gain(L, T, C, P) == want
    assert TP.gain(-np.inf, -16.0, -1.0, 30000.0) == O.UNITY
    assert TP.gain(-np.inf, -16.0, -1.0, 0.0) == O.UNITY
