"""CPU tests of the FLAC format (DESIGN.md 3.5), pinned by two programs that share no code: the oracle encoder
(tests/flac_oracle.c, the contract restated) and an RFC 9639 decoder (tests/flac_decode.c)."""
import numpy as np
import pytest

import flac_codec as F
import resample_oracle as R

RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)
ODD_RATE = 11025   # accepted by the output-rate conversion, no RFC code: 16-bit Hz in the frame header


class Bits:
    def __init__(self):
        self.bits = []

    def put(self, n, v):
        self.bits += [(v >> (n - 1 - i)) & 1 for i in range(n)]

    def pad(self):
        while len(self.bits) % 8:
            self.bits.append(0)

    def data(self):
        assert len(self.bits) % 8 == 0
        return bytes(int("".join(map(str, self.bits[i:i + 8])), 2) for i in range(0, len(self.bits), 8))


def _crc(data, poly, width):
    c, top, mask = 0, 1 << (width - 1), (1 << width) - 1
    for b in data:
        c ^= b << (width - 8)
        for _ in range(8):
            c = ((c << 1) ^ poly) & mask if c & top else (c << 1) & mask
    return c


def test_known_answer_fixed_order_1():
    """x = 0 0 0 10 11 at 22 050 Hz, assembled bit by bit from RFC 9639: one frame of 5 samples, FIXED order 1
    (order sums over sample 4: 11, 1, 9, 19, 29), one partition, Rice k = 2 (4 (k + 1) + sum(u >> k) is 26, 19, 17,
    18, 21 for k = 0..4), residuals 0 0 10 1 -> zigzag 0 0 20 2."""
    x = np.array([0, 0, 0, 10, 11], np.int16)
    fr = Bits()
    fr.put(16, 0xFFF8)
    fr.put(4, 0b0110)       # blocksize: 8 bits of (blocksize - 1) at the end of the header
    fr.put(4, 0b0110)       # 22 050 Hz
    fr.put(4, 0)            # mono
    fr.put(3, 0b100)        # 16 bit
    fr.put(1, 0)
    fr.put(8, 0)            # frame number 0
    fr.put(8, 4)            # blocksize - 1
    fr.put(8, _crc(fr.data(), 0x07, 8))
    fr.put(1, 0)
    fr.put(6, 0b001001)     # FIXED, order 1
    fr.put(1, 0)            # no wasted bits
    fr.put(16, 0)           # warm-up sample
    fr.put(2, 0)            # Rice, 4-bit parameters
    fr.put(4, 0)            # partition order 0
    fr.put(4, 2)            # k = 2
    for u in (0, 0, 20, 2):
        fr.put((u >> 2) + 1, 1)
        fr.put(2, u & 3)
    fr.pad()
    fr.put(16, _crc(fr.data(), 0x8005, 16))
    frame = fr.data()
    st = Bits()
    st.put(32, int.from_bytes(b"fLaC", "big"))
    st.put(1, 1)
    st.put(7, 0)
    st.put(24, 34)
    for n, v in ((16, 4096), (16, 4096), (24, len(frame)), (24, len(frame)), (20, 22050), (3, 0), (5, 15), (36, 5)):
        st.put(n, v)
    st.put(128, 0)
    want = st.data() + frame
    assert len(st.data()) == 42 and len(frame) == 7 + (8 + 16 + 6 + 4 + 17 + 7) // 8 + 2
    got, info = F.decode(want)
    assert np.array_equal(got, x)
    assert info["total_samples"] == 5 and info["min_framesize"] == len(frame)
    assert F.encode(x, 22050) == want


def _check(x, hz=22050):
    data = F.encode(x, hz)
    got, info = F.decode(data)
    assert np.array_equal(got, np.asarray(x, np.int16))
    n = len(x)
    frames = -(-n // 4096)
    assert info["min_blocksize"] == info["max_blocksize"] == 4096
    assert info["sample_rate"] == hz and info["channels"] == 1 and info["bits_per_sample"] == 16
    assert info["total_samples"] == n and info["md5_zero"] == 1
    if frames == 0:
        assert len(data) == 42 and info["min_framesize"] == info["max_framesize"] == 0
    else:
        assert 0 < info["min_framesize"] <= info["max_framesize"] <= F.FRAME_MAX
    assert len(data) <= F.bound(n)
    return data


def _cases():
    rng = np.random.default_rng(9639)
    cases = {}
    for n in (0, 1, 2, 4, 5, 4095, 4096, 4097, 8192, 8193):
        cases[f"len{n}"] = np.clip(np.cumsum(rng.integers(-300, 301, n)), -32768, 32767).astype(np.int16)
    cases["zeros"] = np.zeros(9000, np.int16)
    cases["constant"] = np.full(8192 + 100, -1234, np.int16)
    alt = np.empty(8200, np.int16)
    alt[0::2], alt[1::2] = 32767, -32768
    cases["alternation"] = alt
    cases["alternation_32767"] = np.where(np.arange(4100) % 2, -32767, 32767).astype(np.int16)
    cases["white_noise"] = rng.integers(-32768, 32768, 5 * 4096 + 77).astype(np.int16)
    cases["ramp"] = (np.arange(12000) * 5 - 30000).astype(np.int16)
    last = np.full(4096, 77, np.int16)
    last[-1] = 78
    cases["constant_but_last"] = np.concatenate([last, last])
    cases["speechlike"] = (8000 * np.sin(np.arange(20000) * 0.05) + rng.normal(0, 20, 20000)).astype(np.int16)
    return cases


CASES = _cases()


@pytest.mark.parametrize("name", sorted(CASES))
def test_round_trip(name):
    _check(CASES[name])


def test_subframe_kinds():
    # a frame header of 6 bytes at 22 050 Hz (frame 0, 4096 samples); the subframe type follows it
    def kind(data):
        return data[42 + 6] >> 1
    assert kind(F.encode(CASES["zeros"], 22050)) == 0                   # CONSTANT
    assert kind(F.encode(CASES["white_noise"], 22050)) == 1             # VERBATIM
    assert kind(F.encode(CASES["ramp"], 22050)) == 0b001010             # FIXED order 2
    # the ramp's residuals of order 2 are all zero: one bit per sample and a 4-bit parameter
    assert len(F.encode(CASES["ramp"][:4096], 22050)) < 42 + 6 + 1 + 4 + 1 + 4096 // 8 + 8


@pytest.mark.parametrize("hz", RATES + (ODD_RATE,))
def test_rates(hz):
    x = CASES["speechlike"]
    data = _check(x, hz)
    code = data[42 + 2] & 0xF
    assert code == {8000: 4, 16000: 5, 22050: 6, 24000: 7, 32000: 8, 44100: 9, 48000: 10}.get(hz, 13)


def test_corpus_sentences(H, small_db, front_small, oracle_small):
    texts = H.corpus.batch(4, seed=77, target_chars=150)
    speeds = [1.0, 1.0, 0.7, 1.6]
    plan = front_small.plan(texts, speeds)
    prm = front_small.params()
    for u in range(plan.n_utts):
        x = oracle_small.synth(prm, plan.utt_ops(u), speeds[u])[0]
        assert len(x) > 4096
        data = _check(x)
        assert len(data) < 0.8 * 2 * len(x)
        _check(R.resample(x, 16000), 16000)


def test_decoder_rejects_flipped_bits():
    data = bytearray(F.encode(CASES["speechlike"], 22050))
    with pytest.raises(F.DecodeError, match="-5"):        # CRC-8 of the frame header
        bad = bytearray(data)
        bad[42 + 4] ^= 0x01
        F.decode(bytes(bad))
    with pytest.raises(F.DecodeError, match="-6"):        # CRC-16 of the frame
        bad = bytearray(data)
        bad[42 + 200] ^= 0x10
        F.decode(bytes(bad))
    with pytest.raises(F.DecodeError):
        F.decode(b"fLaX" + bytes(data[4:]))
    with pytest.raises(F.DecodeError):
        F.decode(bytes(data[:-1]))


def test_library_bound_covers_every_case(H):
    gpu = H.importlib.import_module("2026-simple-c-tts_b200.gpu")
    L = gpu.lib()
    for name, x in CASES.items():
        b = int(L.ctts_gpu_flac_bound(len(x)))
        assert b == F.bound(len(x))
        assert len(F.encode(x, 22050)) <= b, name
    noise = CASES["white_noise"][:5 * 4096]   # whole frames: VERBATIM everywhere
    assert int(L.ctts_gpu_flac_bound(len(noise))) <= 1.01 * len(F.encode(noise, 22050))


# ---------------------------------------------------------------------------------- frame numbers (RFC 9639 9.1.5)

def _coded_number(v):
    """RFC 9639's coding of a frame number: 7 bits in one byte below 2^7; else a first byte of (extra + 1) one-bits,
    a zero and the top bits, then `extra` bytes 10xxxxxx of six bits each, with extra the least of 1 .. 6 for which
    the value fits 6 + 5 extra bits (11 bits in two bytes, 16 in three, 21 in four)."""
    if v < 0x80:
        return bytes([v])
    extra = next(e for e in range(1, 7) if v < 1 << (5 * e + 6))
    first = (0xFF00 >> (extra + 1)) & 0xFF | v >> (6 * extra)
    return bytes([first] + [0x80 | (v >> (6 * i)) & 0x3F for i in range(extra - 1, -1, -1)])


def test_frame_number_coding_known_answers():
    """A constant signal of 2 049 whole frames and one sample: every frame is CONSTANT (6-byte subframe and CRC), so
    frame f starts at 42 + sum of the earlier frames' 4 + len(code) + 1 + 3 + 2 bytes.  The header bytes of frames
    127, 128, 2047 and 2048 are the RFC's codes, and the decoder reads every number back."""
    assert [_coded_number(v).hex() for v in (127, 128, 2047, 2048, 65535, 65536)] == \
        ["7f", "c280", "dfbf", "e0a080", "efbfbf", "f0908080"]
    n = 2049 * 4096 + 1
    x = np.full(n, 321, np.int16)
    data = F.encode(x, 22050)
    at, starts = 42, []
    for f in range(2050):
        starts.append(at)
        at += 4 + len(_coded_number(f)) + (1 if f == 2049 else 0) + 1 + 3 + 2   # frame 2049: 1 sample, 8-bit blocksize
    assert at == len(data)
    for f, code in ((127, "7f"), (128, "c280"), (2047, "dfbf"), (2048, "e0a080")):
        assert data[starts[f]:starts[f] + 2] == b"\xff\xf8"
        assert data[starts[f] + 4:starts[f] + 4 + len(code) // 2].hex() == code, f
    got, info, rep = F.decode(data, report=True)
    assert np.array_equal(got, x) and info["total_samples"] == n
    assert rep.number.tolist() == list(range(2050))
    assert rep.header_bytes.tolist() == [4 + len(_coded_number(f)) + (f == 2049) + 1 for f in range(2050)]
    assert (rep.kind == F.CONSTANT).all() and rep.blocksize[-1] == 1


# ---------------------------------------------------------------------------------- the device tests' signals

def _rice_bits(z):
    """The least bits of one partition of zigzag residuals: 4-bit parameter, then k + 1 + (u >> k) per residual."""
    return 4 + min(len(z) * (k + 1) + int((z >> k).sum()) for k in range(15))


def _fixed_bits(x, order, po):
    """Partition bits of a FIXED subframe of x with the given order and partition order."""
    r = x.astype(np.int64)
    for _ in range(order):
        r = np.diff(r)
    z = np.where(r >= 0, 2 * r, -2 * r - 1)     # residuals of samples order .. n - 1
    m = len(x) >> po
    return sum(_rice_bits(z[max(j * m - order, 0):(j + 1) * m - order]) for j in range(1 << po))


def _residual_sums(x):
    r, out = x.astype(np.int64), []
    for o in range(5):
        out.append(int(np.abs(r[4 - o:]).sum()))
        r = np.diff(r)
    return out


def test_device_signals_reach_their_decisions():
    """CPU witness of test_gpu_flac_signals.py: the oracle's file of each constructed signal, as the decoder parsed
    it, makes the decision the signal is built for."""
    import edge_voices as E
    reports = {}
    for case, x in E.flac_signals():
        data = F.encode(x, 22050)
        got, _, rep = F.decode(data, report=True)
        assert np.array_equal(got, x)
        assert rep.blocksize.tolist() == [4096] * (len(x) // 4096) + ([len(x) % 4096] if len(x) % 4096 else [])
        reports[case] = (x, data, rep)
    assert reports["constant_then_fixed"][2].kind.tolist() == [F.CONSTANT] * 2 + [F.FIXED] * 2
    x, data, rep = reports["noise"]
    assert (rep.kind == F.VERBATIM).all() and 0.99 * F.bound(len(x)) <= len(data) <= F.bound(len(x))
    rep = reports["half_noise"][2]
    assert (rep.kind == F.FIXED).all() and (rep.kmin == 0).all() and (rep.kmax == 14).all()
    x, _, rep = reports["alternating"]
    r = x.astype(np.int64)
    for _ in range(4):
        r = np.diff(r)
    assert np.abs(r).max() == 16 * 32767 + 8 and (rep.kind == F.VERBATIM).all()   # order-4 zigzag near 2^20
    assert [reports[f"order{d}"][2].order.tolist() for d in range(5)] == [[d] for d in range(5)]
    assert all((reports[f"order{d}"][2].kind == F.FIXED).all() for d in range(5))
    x, _, rep = reports["ramp"]
    assert (rep.kind == F.FIXED).all() and (rep.order == 2).all()
    for f in range(len(rep)):
        s = _residual_sums(x[4096 * f:4096 * (f + 1)])
        assert s[1] > 0 and s[2] == s[3] == s[4] == 0      # orders 2, 3 and 4 tie: the lowest wins
    binding = []
    for r in E.FLAC_LAST:
        x, _, rep = reports[f"last{r}"]
        assert rep.blocksize[-1] == r and (rep.order[:-1] == 4).all()
        last = rep[-1]
        tail = x[-r:]
        assert last.kind == (F.CONSTANT if r == 1 else F.VERBATIM if r <= 8 else F.FIXED)   # few samples: raw is cheaper
        if last.kind == F.FIXED:
            assert last.order == 4 and (r >> last.po) > 4 and r % (1 << last.po) == 0
            # the partition order the rule (n >> po) > order rules out, with m = order samples per partition
            po_out = next((p for p in range(9) if r % (1 << p) == 0 and r >> p == 4), None)
            if po_out is not None and _fixed_bits(tail, 4, po_out) < _fixed_bits(tail, 4, int(last.po)):
                binding.append(r)
    assert 16 in binding, binding     # the rule, not the bit count, decides the last frame's partition order
