"""GPU tests of the loudness normalization (DESIGN.md 3.6) on constructed signals (edge_voices.loudness_signals, fed
through the voice of edge_voices.family_signals, whose native output is the signal itself): output rates where fs / 10
is not a whole number (sub-blocks of fs / 10 and fs / 10 + 1 samples, both scan transitions), lengths at every block
and launch boundary of the loudness kernels, and signals that drive each gate and the gain rule.  test_loudness.py
witnesses on the CPU that every signal reaches its path.  The device's L agrees with the oracle to 1e-6 LU, its G and
its output equal the oracle's.

The clamp of k to +-8000 is out of reach with accepted settings: T is in [-60, -5], an int16 signal measures at most
about +4 LUFS and a defined L is above -70, so k stays within about [-6400, 6500].  No test drives it.

Run on a B200 with:  python -m pytest tests/test_gpu_loudness_signals.py -m gpu
"""
import numpy as np
import pytest

import edge_voices as E
import loudness_oracle as O
import resample_oracle as R
from test_gpu_flac import _check_files, _flac_session
from test_gpu_loudness import _check_ld, _check_pcm, _ctx, _oracle, _slices

pytestmark = pytest.mark.gpu

FLAC_RATE = 8015   # fractional: the FLAC session with loudness on


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


def _session(g, pieces, prm):
    cap = sum(int(((g.bounds(p).astype(np.int64) + 7) // 8 * 8).sum()) for p in pieces) + 64
    buf = np.zeros(cap, np.int16)
    off, cnt = g.synth_pieces(pieces, prm, buf)
    return _slices(buf, off, cnt)


@pytest.mark.parametrize("hz", E.LD_RATES)
def test_signals_match_the_oracle(gpu, hz):
    assert R.ratio(hz) is not None
    fam = E.signal_family(f"loudness_{hz}")
    plan, prm = fam.plan(), fam.prm()
    xs = [R.resample(x, hz) for x in fam.info["signals"]]
    n = plan.n_utts
    for T, C in E.LD_SETTINGS:
        want = _oracle(xs, hz, T, C)
        assert any(G == O.UNITY and np.isfinite(L) for _, L, G in want) and any(G != O.UNITY for _, _, G in want)
        g = _ctx(gpu, fam.db, hz, T, C)
        try:
            what = f"{hz} Hz, T {T}"
            rp = g.create_plan(plan, prm)
            for run in range(2):
                rp.run()
                lufs, gain = rp.loudness()
                ties = _check_ld(lufs, gain, want, T, f"{what} resident run {run}")
                _check_pcm(rp.utterances(), want, ties, f"{what} resident run {run}")
            rp.close()
            pcm, off, cnt = g.synth_batch(plan, prm)
            _check_pcm(_slices(pcm, off, cnt), want, ties, f"{what} synth_batch")
            pieces = [plan.select(range(0, n // 3)), plan.select(range(n // 3, n))]
            _check_pcm(_session(g, pieces, prm), want, ties, f"{what} session")
            if hz == FLAC_RATE:
                assert not ties
                _check_files(*_flac_session(g, pieces, prm), [y for y, _, _ in want], hz, f"{what} FLAC session")
        finally:
            g.close()


@pytest.mark.parametrize("hz", (22050, 11025))
def test_long_utterance(gpu, hz):
    """6.3 minutes, thousands of chunks: the scan's longest serial chain."""
    fam = E.signal_family("long")
    plan, prm = fam.plan(), fam.prm()
    x = fam.info["signals"][0]
    y = x if hz == 22050 else R.resample(x, hz)
    assert len(y) * 10 // hz > 3000
    for T, C in E.LD_SETTINGS:
        want = _oracle([y], hz, T, C)
        g = _ctx(gpu, fam.db, hz, T, C)
        try:
            rp = g.create_plan(plan, prm)
            rp.run()
            lufs, gain = rp.loudness()
            ties = _check_ld(lufs, gain, want, T, f"long {hz} T {T}")
            _check_pcm(rp.utterances(), want, ties, f"long {hz} T {T}")
            rp.close()
        finally:
            g.close()
