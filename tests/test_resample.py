"""CPU tests of the output-rate conversion (DESIGN.md 3.4): the filter and the oracle against scipy, the product's
host tap table against the oracle, and the output-length rule."""
import ctypes as C
import importlib
import math

import numpy as np
import pytest

import resample_oracle as R

scipy_signal = pytest.importorskip("scipy.signal")

RATES = [hz for hz in R.COMMON_RATES if hz != R.NATIVE]
BETA = 0.1102 * (70 - 8.7)


def _scipy_taps(hz):
    L, M = R.ratio(hz)
    N = 2 * R.H_ZERO_CROSSINGS * max(L, M) + 1
    return L * scipy_signal.firwin(N, 0.94 / max(L, M), window=("kaiser", BETA))


def _ulps(a, b):
    a = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(a - b)


def test_ratio_rules():
    for hz in R.COMMON_RATES:
        L, M = R.ratio(hz)
        assert math.gcd(L, M) == 1 and L * R.NATIVE == M * hz
    for hz in (7999, 48001, 0, 44099, 47999, 8009):
        assert R.ratio(hz) is None, hz
    accepted = [hz for hz in range(8000, 48001) if R.ratio(hz) is not None]
    for hz in accepted[::97]:
        L, M = R.ratio(hz)
        assert max(L, M) <= 1024


@pytest.mark.parametrize("hz", RATES)
def test_oracle_taps_equal_firwin(hz):
    g = R.taps(hz)
    assert _ulps(g, _scipy_taps(hz).astype(np.float32)).max() <= 1


@pytest.mark.parametrize("hz", RATES)
def test_product_taps_equal_oracle(hz):
    """The tap table libctts_gpu.so uploads is computed on the host (csrc/gpu/ctts_tables.c): no device needed."""
    gpu = importlib.import_module("2026-simple-c-tts_b200.gpu")
    lib = gpu.lib()
    L, M = R.ratio(hz)
    g = np.zeros(2 * 40 * max(L, M) + 1, np.float32)
    lib.ctts_host_resample_taps.argtypes = [C.c_uint, C.c_uint, C.c_void_p]
    lib.ctts_host_resample_taps.restype = None
    lib.ctts_host_resample_taps(L, M, g.ctypes.data)
    assert _ulps(g, R.taps(hz)).max() <= 1


@pytest.mark.parametrize("hz", RATES)
def test_filter_response(hz):
    L, M = R.ratio(hz)
    g = R.taps(hz).astype(np.float64) / L
    f_low = min(R.NATIVE, hz)
    fs = R.NATIVE * L   # the rate the filter runs at
    w_pass = np.linspace(0, 0.44 * f_low, 400)
    w_stop = np.linspace(0.5 * f_low, fs / 2, 4000)
    _, hp = scipy_signal.freqz(g, worN=w_pass, fs=fs)
    _, hs = scipy_signal.freqz(g, worN=w_stop, fs=fs)
    ripple = 20 * np.log10(np.abs(hp))
    assert np.abs(ripple).max() <= 0.005, ripple.max()
    # 70.0 dB from 0.5 f_low on; the 161-tap filters of R = 2 (11 025 and 44 100 Hz) reach 69.4 dB
    assert 20 * np.log10(np.abs(hs).max()) <= (-69.4 if max(L, M) <= 2 else -70.0)


def _resample_poly_int16(x, hz):
    L, M = R.ratio(hz)
    h = R.taps(hz).astype(np.float64) / L
    y = scipy_signal.resample_poly(x.astype(np.float64), L, M, window=h)
    return np.clip(np.rint(y), -32768, 32767)


def _inputs(rng):
    yield rng.integers(-12000, 12000, 4000).astype(np.int16)                      # random
    t = np.arange(3000)
    yield np.where((t // 37) % 2 == 0, 32767, -32768).astype(np.int16)           # full-scale square: saturation
    yield np.where((t // 5) % 2 == 0, 32767, -32768).astype(np.int16)
    imp = np.zeros(2500, np.int16)
    imp[[0, 1, 700, 2499]] = [32767, -32768, 20000, 32767]
    yield imp                                                                     # impulses, also at both ends


@pytest.mark.parametrize("hz", RATES)
def test_oracle_within_one_lsb_of_scipy(hz):
    rng = np.random.default_rng(hz)
    for x in _inputs(rng):
        y = R.resample(x, hz)
        z = _resample_poly_int16(x, hz)
        assert len(y) == len(z) == R.count(hz, len(x))
        assert np.abs(y.astype(np.int64) - z).max() <= 1


@pytest.mark.parametrize("hz", RATES)
def test_oracle_every_short_length(hz):
    rng = np.random.default_rng(7 + hz)
    lengths = list(range(0, 2 * R.H_ZERO_CROSSINGS + 4)) + [1000, 2047, 3001]
    for n in lengths:
        x = rng.integers(-32768, 32768, n).astype(np.int16)
        y = R.resample(x, hz)
        L, M = R.ratio(hz)
        assert len(y) == -(-n * L // M)
        if n:
            z = _resample_poly_int16(x, hz)
            assert len(z) == len(y) and np.abs(y.astype(np.int64) - z).max() <= 1, n


@pytest.mark.parametrize("hz", R.COMMON_RATES)
def test_count_rule(hz):
    L, M = R.ratio(hz)
    for n in range(0, 5001):
        assert R.count(hz, n) == -(-n * L // M)
    assert R.count(hz, 0) == 0


def test_capacity_hint_rate_scales(front_small):
    pipe = importlib.import_module("2026-simple-c-tts_b200.pipeline")
    batch = pipe.TextBatch(["olá mundo", "Bom dia, como vai? 12 casas!", ""], [1.0, 0.7, 1.3])
    native = pipe.capacity_hint(front_small, batch)
    assert pipe.capacity_hint(front_small, batch, 22050) == native
    for hz in RATES:
        L, M = R.ratio(hz)
        got = pipe.capacity_hint(front_small, batch, hz)
        assert got >= -(-native * L // M)


def test_rate_headers_are_exported(H):
    """ctts_gpu_set_output_rate (ctts_gpu.h) and ctts_b200_rate.h load from the libraries without a device."""
    import os
    import re
    pipe = importlib.import_module("2026-simple-c-tts_b200.pipeline")
    gpu = importlib.import_module("2026-simple-c-tts_b200.gpu")
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(H.ROOT, "include", "ctts_b200_rate.h")).read(), flags=re.S)
    names = sorted(set(re.findall(r"\b(ctts_b200_[a-z0-9_]+)\s*\(", text)))
    assert names == ["ctts_b200_capacity_hint_rate"]
    assert hasattr(pipe.lib(), names[0]) and hasattr(gpu.lib(), "ctts_gpu_set_output_rate")
