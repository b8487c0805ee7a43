"""CPU tests of the loudness normalization (DESIGN.md 3.6): the product's host coefficients against BS.1770-4 and the
oracle, the oracle's loudness against an independent scipy restatement, known answers, the gain table and the gain
rule."""
import ctypes as C
import importlib

import numpy as np
import pytest

import loudness_oracle as O

S = pytest.importorskip("scipy.signal")

RATES = (8000, 11025, 16000, 22050, 44100, 48000)
# ITU-R BS.1770-4, tables 1 and 2 (48 kHz)
BS1770_SHELF_B = (1.53512485958697, -2.69169618940638, 1.19839281085285)
BS1770_SHELF_A = (1.0, -1.69065929318241, 0.73248077421585)
BS1770_HP_A = (1.0, -1.99004745483398, 0.99007225036621)


def _product(fs):
    lib = importlib.import_module("2026-simple-c-tts_b200.gpu").lib()
    lib.ctts_host_loudness_filter.argtypes = [C.c_uint, C.c_void_p, C.c_void_p]
    lib.ctts_host_loudness_filter.restype = None
    shelf, hp = np.zeros(5), np.zeros(2)
    lib.ctts_host_loudness_filter(fs, shelf.ctypes.data, hp.ctypes.data)
    return shelf, hp


def _scipy_lufs(x, fs):
    """BS.1770-4 restated with scipy.signal.lfilter, independently of the oracle."""
    sb, sa, hb, ha = O.filter_coeffs(fs)
    y = S.lfilter(hb, ha, S.lfilter(sb, sa, np.asarray(x, np.float64) / 32768.0))
    starts = [k * fs // 10 for k in range(len(y) * 10 // fs + 2)]
    subs = [k for k in range(len(starts) - 1) if starts[k + 1] <= len(y)]
    if len(subs) < 4:
        return -np.inf
    y2 = y * y
    z = np.array([y2[starts[j]:starts[j + 4]].mean() for j in range(len(subs) - 3)])
    z1 = z[z > 10 ** ((-70 + 0.691) / 10)]
    if not len(z1):
        return -np.inf
    z2 = z1[z1 > z1.mean() / 10]
    return -0.691 + 10 * np.log10(z2.mean())


def _sine(fs, seconds, amp, f=997.0):
    t = np.arange(int(round(seconds * fs))) / fs
    return np.round(amp * np.sin(2 * np.pi * f * t)).astype(np.int16)


def test_product_coefficients_equal_bs1770_at_48k():
    shelf, hp = _product(48000)
    assert np.abs(shelf[:3] - BS1770_SHELF_B).max() <= 1e-12
    assert np.abs(shelf[3:] - BS1770_SHELF_A[1:]).max() <= 1e-12
    assert np.abs(hp - BS1770_HP_A[1:]).max() <= 1e-12


@pytest.mark.parametrize("fs", RATES)
def test_product_coefficients_equal_oracle(fs):
    shelf, hp = _product(fs)
    sb, sa, hb, ha = O.filter_coeffs(fs)
    assert shelf.tobytes() == np.concatenate([sb, sa[1:]]).tobytes()
    assert hp.tobytes() == ha[1:].tobytes()
    assert list(hb) == [1.0, -2.0, 1.0] and sa[0] == ha[0] == 1.0


def _inputs():
    rng = np.random.default_rng(7)
    yield "sine 22050", _sine(22050, 3.0, 8000, 440.0), 22050
    yield "sine 8000", _sine(8000, 2.5, 20000, 1000.0), 8000
    yield "noise 16000", np.clip(rng.normal(0, 3000, 16000 * 3), -32768, 32767).astype(np.int16), 16000
    yield "noise 48000", np.clip(rng.normal(0, 300, 48000 * 2), -32768, 32767).astype(np.int16), 48000
    loud, quiet = _sine(22050, 3.0, 16000), _sine(22050, 3.0, 80)
    yield "two-level 22050", np.concatenate([loud, quiet]), 22050
    yield "sine 11025", _sine(11025, 2.77, 12000, 300.0), 11025
    yield "noise 11025", np.clip(rng.normal(0, 5000, 11025 * 2 + 517), -32768, 32767).astype(np.int16), 11025


@pytest.mark.parametrize("name,x,fs", list(_inputs()), ids=[n for n, _, _ in _inputs()])
def test_oracle_equals_scipy(name, x, fs):
    got, want = O.lufs(x, fs), _scipy_lufs(x, fs)
    assert np.isfinite(got) and abs(got - want) <= 1e-9, (name, got, want)


def test_relative_gate_removes_the_quiet_half():
    loud, quiet = _sine(22050, 3.0, 16000), _sine(22050, 3.0, 80)
    both = O.lufs(np.concatenate([loud, quiet]), 22050)
    # the quiet half is 46 dB down: gated away, apart from the blocks that straddle the step
    assert abs(both - O.lufs(loud, 22050)) < 0.5
    assert both > O.lufs(loud, 22050) - 3.0 + 1.0


@pytest.mark.parametrize("fs", (8000, 11025, 16000, 22050, 48000))
def test_undefined_loudness(fs):
    short = _sine(fs, 1.0, 10000)[: (4 * fs) // 10 - 1]      # 399 ms (one sample short of a block)
    assert O.lufs(short, fs) == -np.inf and _scipy_lufs(short, fs) == -np.inf
    block = _sine(fs, 1.0, 10000)[: (4 * fs) // 10]           # exactly one block
    assert np.isfinite(O.lufs(block, fs)) and abs(O.lufs(block, fs) - _scipy_lufs(block, fs)) <= 1e-9
    assert O.lufs(np.zeros(fs * 2, np.int16), fs) == -np.inf
    assert O.lufs(np.zeros(0, np.int16), fs) == -np.inf
    faint = _sine(fs, 2.0, 2)                                 # about -87 LUFS: below the absolute gate
    assert O.lufs(faint, fs) == -np.inf and _scipy_lufs(faint, fs) == -np.inf
    y, L, G = O.normalize(faint, fs, -16.0, -1.0)
    assert G == O.UNITY and np.array_equal(y, faint)


@pytest.mark.parametrize("fs,tol", [(48000, 0.01), (44100, 0.01), (22050, 0.05), (16000, 0.05), (11025, 0.05), (8000, 0.05)])
def test_full_scale_997hz_reads_minus_3(fs, tol):
    x = _sine(fs, 10.0, 32767)
    assert abs(O.lufs(x, fs) - (-3.01)) <= tol


def test_product_gain_table_equals_oracle():
    lib = importlib.import_module("2026-simple-c-tts_b200.gpu").lib()
    lib.ctts_host_loudness_gains.argtypes = [C.c_void_p]
    lib.ctts_host_loudness_gains.restype = None
    t = np.zeros(2 * O.K_MAX + 1, np.uint32)
    lib.ctts_host_loudness_gains(t.ctypes.data)
    assert np.array_equal(t, O.table())
    assert t[O.K_MAX] == O.UNITY and t[-1] == 655360000
    lib.ctts_host_loudness_ceiling.argtypes = [C.c_float]
    lib.ctts_host_loudness_ceiling.restype = C.c_uint
    for c in (0.0, -0.1, -1.0, -3.0, -20.0):
        assert lib.ctts_host_loudness_ceiling(c) == O.ceiling(c)
    assert O.ceiling(0.0) == 32767 and O.ceiling(-20.0) == 3276


@pytest.mark.parametrize("c", (0.0, -20.0))
def test_gain_rule_holds_the_ceiling(c):
    fs = 16000
    full = _sine(fs, 2.0, 32767)
    full[100] = -32768
    square = np.where(_sine(fs, 2.0, 1000, 50.0) >= 0, 32767, -32768).astype(np.int16)
    for x in (full, square):
        for target in (-5.0, -16.0, -60.0):
            y, L, G = O.normalize(x, fs, target, c)
            assert np.isfinite(L)
            assert np.abs(y.astype(np.int32)).max() <= O.ceiling(c)
            assert G == min(O.table()[int(np.clip(np.floor(100 * (target - L) + 0.5), -8000, 8000)) + O.K_MAX],
                            O.ceiling(c) * 65536 // 32768)


def test_unity_gain_is_the_identity():
    rng = np.random.default_rng(3)
    x = rng.integers(-32768, 32768, 50000).astype(np.int16)
    assert np.array_equal(((x.astype(np.int64) * O.UNITY + 32768) >> 16).astype(np.int16), x)
    q = _sine(22050, 2.0, 1000)
    L = O.lufs(q, 22050)
    y, L2, G = O.normalize(q, 22050, float(np.float32(L)), 0.0)   # a target equal to L: k = 0
    assert G == O.UNITY and np.array_equal(y, q) and L2 == L


def test_target_reached_within_a_step():
    fs = 22050
    x = np.concatenate([_sine(fs, 2.0, 3000, 300.0), _sine(fs, 1.5, 6000, 2000.0)])
    for target in (-16.0, -23.0, -30.0):
        y, L, G = O.normalize(x, fs, target, 0.0)
        assert abs(O.lufs(y, fs) - target) < 0.05
