"""What time_stretch does to a steady harmonic tone (DESIGN.md 3.2, "What the stretch does to pitch").

At its fixed point the WSOLA chain keeps every frame at its nominal analysis position, so time_stretch is unaligned
overlap-add: frames taken every 128 samples are laid down every `hop` samples and their phases jump from frame to frame.
The result is an inharmonic comb, with lines at f_k 128 / hop + m fs / hop (f_k the tone's harmonics) weighted by the
window's spectrum.  It is not the tone at a new pitch.  Resampling that by 128 / hop, the usual way to turn a stretch into
a pitch shift that keeps the duration, puts the lines at f_k + m fs / 128, the tone's own harmonics and their sidebands
at the frame rate.  There is nothing at the shifted fundamental 120 hop / 128 Hz.

The stretch is examined at every hop 64 .. 256 through tests/stretch_hop_oracle.c, the oracle's loop at a given hop.
That loop is checked bit for bit against ctts_oracle_time_stretch at the hops a speed reaches.
"""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

import resample_oracle as R

scipy_signal = pytest.importorskip("scipy.signal")

FS = 22050
F0 = 120.0
NFFT = 1 << 20


def _tone(seconds=2.0):
    t = np.arange(int(seconds * FS)) / FS
    x = sum(np.sin(2 * np.pi * k * F0 * t + k) / k for k in range(1, 9))
    return (x / np.abs(x).max() * 12000).astype(np.int16)


def _spectrum(y):
    s = np.abs(np.fft.rfft(y.astype(np.float64) * np.hanning(len(y)), NFFT))
    return s, np.arange(len(s)) * FS / NFFT


def _dominant(s, f, lo=30.0, hi=2000.0):
    """(frequency, magnitude) of the strongest line in [lo, hi]."""
    sel = np.nonzero((f > lo) & (f < hi))[0]
    k = sel[np.argmax(s[sel])]
    return f[k], s[k]


def _db_at(s, f, freq, ref):
    """Level of the spectrum at freq (the largest bin within 0.1 Hz) relative to ref, in dB."""
    sel = np.abs(f - freq) <= 0.1
    return 20 * np.log10(s[sel].max() / ref)


def _comb_distance(freq, base, step):
    """Distance from freq to the nearest k base + m step, k = 1 .. 8, m any integer."""
    return min(abs((freq - k * base) - round((freq - k * base) / step) * step) for k in range(1, 9))


@pytest.fixture(scope="module")
def stretch(H, oracle_small, tmp_path_factory):
    """stretch(x, hop) -> (v, frames): the oracle's time_stretch loop at synthesis hop `hop`."""
    so = str(tmp_path_factory.mktemp("stretch_hop") / "libstretch_hop_oracle.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stretch_hop_oracle.c")
    subprocess.run([shutil.which("gcc") or "cc", "-O2", "-std=c99", "-ffp-contract=off", "-Wall", "-Wextra", "-fPIC", "-shared",
                    "-o", so, src], check=True)
    L = C.CDLL(so)
    L.stretch_hop_oracle_stretch_cap.argtypes = [C.c_size_t, C.c_uint32]
    L.stretch_hop_oracle_stretch_cap.restype = C.c_size_t
    L.stretch_hop_oracle_stretch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                             C.POINTER(C.c_uint32)]
    L.stretch_hop_oracle_stretch.restype = C.c_int64
    hann = np.ascontiguousarray(oracle_small.tables()[2], np.float32)
    offset = C.cast(H.oracle_lib().ctts_oracle_wsola_offset, C.c_void_p)

    def run(x, hop):
        x = np.ascontiguousarray(x, np.int16)
        y = np.zeros(L.stretch_hop_oracle_stretch_cap(len(x), hop), np.int16)
        fr = C.c_uint32()
        n = L.stretch_hop_oracle_stretch(offset, hann.ctypes.data, x.ctypes.data, len(x), hop, y.ctypes.data, C.byref(fr))
        assert n >= 0
        return y[:n].copy(), int(fr.value)
    return run


def _oracle_stretch(H, oracle, x, speed):
    L = H.oracle_lib()
    o = C.POINTER(C.c_int16)()
    n = C.c_size_t()
    fr = C.c_uint32()
    assert L.ctts_oracle_time_stretch(oracle._h, x.ctypes.data, len(x), C.c_float(speed), C.byref(o), C.byref(n), C.byref(fr)) == 0
    v = np.ctypeslib.as_array(o, shape=(max(n.value, 1),))[:n.value].copy()
    L.ctts_oracle_free(o)
    return v, int(fr.value)


def _speed_for(h):
    """A float32 speed whose time_stretch hop (size_t)(128 / speed) is h, outside the plain-copy band; None if none."""
    for frac in (0.5, 0.25, 0.75, 0.1, 0.9):
        sp = np.float32(128 / (h + frac))
        if int(np.float32(128) / sp) == h and abs(float(sp) - 1) >= 0.01:
            return float(sp)
    return None


def test_hop_loop_is_the_oracle(H, oracle_small, stretch):
    """At the hops a speed reaches, the hop-driven loop is ctts_oracle_time_stretch bit for bit."""
    rng = np.random.default_rng(8)
    x = (rng.normal(0, 3000, 9000) * np.sin(np.arange(9000) / 300.0)).astype(np.int16)
    for h in (64, 70, 100, 126, 129, 150, 200, 256):
        want, fr = _oracle_stretch(H, oracle_small, x, _speed_for(h))
        got, frames = stretch(x, h)
        assert frames == fr == (len(x) - 512) // 128 + 1 and np.array_equal(got, want), h
    assert _speed_for(127) is None   # hops next to 128 are reached by the hop alone
    for n in (0, 100, 511):
        assert len(stretch(x[:n], 127)[0]) == 0


@pytest.mark.parametrize("speed,hop,dominant,tape_db", [(2.0, 64, 3 * 240 - FS / 64, -20), (0.5, 256, 60 + FS / 256, -6)])
def test_speed_makes_a_comb_not_a_new_pitch(H, oracle_small, speed, hop, dominant, tape_db):
    """The speed path itself: the strongest line is a comb line, not the tone moved by the speed factor."""
    v, _ = _oracle_stretch(H, oracle_small, _tone(), speed)
    s, f = _spectrum(v)
    fd, ref = _dominant(s, f)
    assert abs(fd - dominant) < 0.1, (speed, fd, dominant)   # 375.5 Hz at speed 2.0, 146.1 Hz at speed 0.5
    assert _comb_distance(fd, F0 * 128 / hop, FS / hop) < 0.1
    assert _db_at(s, f, F0 * 128 / hop, ref) < tape_db, speed   # 240 Hz / 60 Hz, the "tape" pitch, well below it


def test_stretch_then_resample_never_reaches_the_shifted_pitch(stretch):
    """Every hop: stretched, then resampled by 128 / hop (scipy's polyphase resampler).  The strongest line is one of the
    tone's harmonics or a frame-rate sideband of one (f_k + m fs / 128).  Wherever the would-be fundamental 120 hop / 128
    Hz lies at least 2 Hz from those lines, it is more than 45 dB below the strongest line."""
    x = _tone()
    clear = 0
    for h in range(64, 257):
        if h == 128:
            continue
        v, _ = stretch(x, h)
        g = math.gcd(128, h)
        y = scipy_signal.resample_poly(v.astype(np.float64), 128 // g, h // g)
        assert abs(len(y) - len(x)) <= 1024, h   # the duration is kept
        s, f = _spectrum(y)
        fd, ref = _dominant(s, f)
        assert _comb_distance(fd, F0, FS / 128) < 0.1, (h, fd)
        shifted = F0 * h / 128
        if _comb_distance(shifted, F0, FS / 128) >= 2.0:
            clear += 1
            assert _db_at(s, f, shifted, ref) < -45, (h, _db_at(s, f, shifted, ref))
    assert clear >= 150


@pytest.mark.parametrize("speed,hop,hz", [(2.0, 64, 44100), (0.5, 256, 11025)])
def test_the_project_resampler_agrees(H, oracle_small, speed, hop, hz):
    """At the two hops where a speed and an accepted output rate have the ratio 128 / hop, the project's own rate
    oracle gives the same picture: the strongest line is on the tone's comb, and at hop 64 the shifted fundamental
    (60 Hz, not on the comb) is more than 45 dB below it."""
    assert R.ratio(hz) == ((2, 1) if hop == 64 else (1, 2))
    x = _tone()
    y = R.resample(_oracle_stretch(H, oracle_small, x, speed)[0], hz)
    assert abs(len(y) - len(x)) <= 1024
    s, f = _spectrum(y)
    fd, ref = _dominant(s, f)
    assert _comb_distance(fd, F0, FS / 128) < 0.1, fd
    if hop == 64:
        assert _db_at(s, f, F0 * hop / 128, ref) < -45
