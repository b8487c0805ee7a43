"""CPU tests of the G.711 contract (DESIGN.md 3.7): the oracle's code tables against the pinned SHA-256 values and anchors
(computed from CPython's audioop, which Python 3.13 removes), against audioop itself where it can still be imported, and
the 58-byte header of the .wav files the command line writes (csrc/cli/g711_wav.h), parsed field by field."""
import hashlib
import os
import shutil
import subprocess
import warnings

import numpy as np
import pytest

import g711_oracle as G

SHA256 = {G.ULAW: "81d633c9e6972a18c74a58720b96cb8ca0bdd096d4060b646dd708c3b846019a",
          G.ALAW: "38488f6fd710f4686360edc4d38639f96c491595ef93f8eb8d62d5e07ca6ce7b"}
ANCHORS = {0: (0xFF, 0xD5), -1: (0x7E, 0x55), 100: (0xF2, 0xD3), -100: (0x72, 0x53), 32767: (0x80, 0xAA),
           -32768: (0x00, 0x2A)}


@pytest.mark.parametrize("law", (G.ULAW, G.ALAW))
def test_tables_match_the_pinned_hashes(law):
    t = G.table(law)
    assert t.shape == (65536,) and t.dtype == np.uint8
    assert hashlib.sha256(t.tobytes()).hexdigest() == SHA256[law]


def test_anchor_values():
    for x, (mu, a) in ANCHORS.items():
        assert int(G.lin2ulaw([x])[0]) == mu, x
        assert int(G.lin2alaw([x])[0]) == a, x
        assert int(G.table(G.ULAW)[x + 32768]) == mu and int(G.table(G.ALAW)[x + 32768]) == a, x
    assert G.SILENCE[G.ULAW] == int(G.lin2ulaw([0])[0]) and G.SILENCE[G.ALAW] == int(G.lin2alaw([0])[0])


def test_tables_equal_audioop():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        try:
            import audioop
        except ImportError:
            pytest.skip("audioop is not available (removed in Python 3.13); the pinned hashes stand for it")
    x = np.arange(-32768, 32768, dtype="<i2").tobytes()
    assert audioop.lin2ulaw(x, 2) == G.table(G.ULAW).tobytes()
    assert audioop.lin2alaw(x, 2) == G.table(G.ALAW).tobytes()


def test_packed_layout_pads_with_silence():
    pcm = [np.zeros(0, np.int16), np.array([1, -1, 30000], np.int16), np.arange(8, dtype=np.int16) * 1000]
    for law in (G.ULAW, G.ALAW):
        b = G.packed(pcm, law)
        assert len(b) == 0 + 8 + 8
        assert b[3:8] == bytes([G.SILENCE[law]]) * 5
        assert b[8:16] == G.encode(pcm[2], law).tobytes()


@pytest.fixture(scope="module")
def header_tool(H, tmp_path_factory):
    """A driver that prints g711_wav_header(law, rate, count) in hex, compiled from the product's header."""
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        pytest.skip("no C compiler")
    d = tmp_path_factory.mktemp("g711wav")
    src = d / "hdr.c"
    src.write_text('#include <stdio.h>\n#include <stdlib.h>\n#include "g711_wav.h"\n'
                   "int main(int argc, char** argv) {\n"
                   "    (void)argc;\n"
                   "    uint8_t h[G711_WAV_HEADER_BYTES];\n"
                   "    g711_wav_header(h, atoi(argv[1]), (uint32_t)strtoul(argv[2], NULL, 10), (uint32_t)strtoul(argv[3], NULL, 10));\n"
                   "    for (int i = 0; i < G711_WAV_HEADER_BYTES; i++) printf(\"%02x\", h[i]);\n"
                   "    return 0;\n}\n")
    exe = d / "hdr"
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(H.ROOT, "include"),
                    "-I", os.path.join(H.ROOT, "2026-simple-c-tts_b200", "csrc", "cli"), str(src), "-o", str(exe)], check=True)
    return lambda law, rate, count: bytes.fromhex(subprocess.run([str(exe), str(law), str(rate), str(count)],
                                                                 capture_output=True, text=True, check=True).stdout)


@pytest.mark.parametrize("law,rate,count", [(G.ULAW, 8000, 0), (G.ULAW, 8000, 8000), (G.ALAW, 8000, 12345),
                                            (G.ALAW, 22050, 1), (G.ULAW, 16000, 65537)])
def test_wav_header(header_tool, law, rate, count):
    h = header_tool(law, rate, count)
    assert len(h) == 58
    payload = np.random.default_rng(count).integers(0, 256, count).astype(np.uint8).tobytes()
    f = h + payload + b"\0" * (count & 1)
    info = G.parse_wav(f)
    assert info["law"] == law and info["rate"] == rate and info["count"] == count
    assert info["codes"].tobytes() == payload
    # the fields one by one, at their offsets
    le = lambda a, b: int.from_bytes(h[a:b], "little")
    assert h[:4] == b"RIFF" and le(4, 8) == 50 + count + (count & 1) and h[8:16] == b"WAVEfmt "
    assert le(16, 20) == 18 and le(20, 22) == (7 if law == G.ULAW else 6) and le(22, 24) == 1
    assert le(24, 28) == rate and le(28, 32) == rate and le(32, 34) == 1 and le(34, 36) == 8 and le(36, 38) == 0
    assert h[38:42] == b"fact" and le(42, 46) == 4 and le(46, 50) == count
    assert h[50:54] == b"data" and le(54, 58) == count
