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
