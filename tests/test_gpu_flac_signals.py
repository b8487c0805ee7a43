"""GPU tests of the FLAC output (DESIGN.md 3.5) on constructed signals (edge_voices.flac_signals, fed through the voice
of edge_voices.family_signals, whose native output is the signal itself): every subframe kind, Rice parameters 0 .. 14
in one frame, each fixed order, an order tie, short last frames, a 16-bit rate code, frame numbers coded in three
bytes, and pieces past the byte-offset scan's 1 024-utterance pass and past grid.y = 65 535.  test_flac.py witnesses
on the CPU, from the decoder's frame report, that every signal reaches its decision.  Every file is byte-identical to
the oracle encoder's and decodes to the signal (resampled at other rates).

Run on a B200 with:  python -m pytest tests/test_gpu_flac_signals.py -m gpu
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import edge_voices as E
import flac_codec as F
import resample_oracle as R
from test_gpu_flac import _check_files, _flac_session

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu(H):
    return H.importlib.import_module("2026-simple-c-tts_b200.gpu")


@pytest.mark.parametrize("hz", (22050, 8015))
def test_signals_match_the_oracle(gpu, hz):
    fam = E.signal_family("flac")
    plan, prm = fam.plan(), fam.prm()
    pcm = [x if hz == 22050 else R.resample(x, hz) for x in fam.info["signals"]]
    g = gpu.GpuSynth(fam.db, 0)
    try:
        g.set_output_rate(hz)
        n = plan.n_utts
        pieces = [plan.select(range(0, 5)), plan.select(range(5, n))]
        files = _check_files(*_flac_session(g, pieces, prm), pcm, hz, f"signals {hz} Hz")
    finally:
        g.close()
    for f in files:
        assert f[42 + 2] & 0xF == (6 if hz == 22050 else 13)
    if hz == 22050:   # all VERBATIM: the size bound is tight
        case = [c for c, _ in E.flac_signals()].index("noise")
        assert 0.99 * F.bound(len(pcm[case])) <= len(files[case]) <= F.bound(len(pcm[case]))


def test_frame_numbers_past_2047(gpu):
    """2 049 whole frames and a partial one: frame numbers coded in one, two and three bytes, and the STREAMINFO
    total of 8.4 million samples."""
    fam = E.signal_family("long")
    plan, prm = fam.plan(), fam.prm()
    x = fam.info["signals"][0]
    g = gpu.GpuSynth(fam.db, 0)
    try:
        files = _check_files(*_flac_session(g, [plan], prm), [x], 22050, "2 050 frames")
    finally:
        g.close()
    _, info, rep = F.decode(files[0], report=True)
    assert info["total_samples"] == len(x) and rep.number.tolist() == list(range(E.LONG_FRAMES + 1))
    assert rep.header_bytes[[127, 128, 2047, 2048]].tolist() == [6, 7, 7, 8]


def test_piece_sizes(gpu):
    """One piece of 2 000 utterances (the byte-offset scan carries across 1 024-utterance passes) and one of 70 000
    (the analysis and emission grids split at 65 535).  Every file's offset, size and padding is checked; the bytes of
    the files around both limits and of the last 300 against the oracle, encoded once per distinct signal."""
    fam = E.signal_family("pieces")
    plan, prm = fam.plan(), fam.prm()
    sig = E.piece_signals()
    a = E.PIECE_SIZES[0]
    n = plan.n_utts
    g = gpu.GpuSynth(fam.db, 0)
    try:
        out, off, nbytes, cnt, used = _flac_session(g, [plan.select(range(0, a)), plan.select(range(a, n))], prm)
    finally:
        g.close()
    with ThreadPoolExecutor(max(1, min(8, os.cpu_count() or 1))) as ex:
        want = list(ex.map(lambda x: F.encode(x, 22050), sig))
    size = np.array([len(w) for w in want], np.int64)[np.arange(n) % len(sig)]
    length = np.array([len(x) for x in sig], np.int64)[np.arange(n) % len(sig)]
    assert np.array_equal(nbytes.astype(np.int64), size) and np.array_equal(cnt.astype(np.int64), length)
    ends = off.astype(np.int64) + size
    pads = (ends + 15) // 16 * 16
    assert off[0] == 0 and np.array_equal(off[1:].astype(np.int64), pads[:-1]) and used == pads[-1]
    gaps = np.concatenate([np.arange(e, p) for e, p in zip(ends, pads)])
    assert not out[gaps].any(), "alignment padding is not zero"
    check = sorted({*range(1020, 1030), *range(a + 65530, a + 65540), *range(n - 300, n)})
    for u in check:
        got = out[int(off[u]):int(off[u]) + int(nbytes[u])].tobytes()
        assert got == want[u % len(sig)], f"piece file of utterance {u}"
