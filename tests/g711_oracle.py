"""TEST oracle of the G.711 output (DESIGN.md 3.7, ctts_gpu.h): the ITU-T G.711 reference encoder as the G.191 software
tools and Sun's g711.c state it (CPython 3.12's audioop.lin2ulaw / lin2alaw compute the same on 16-bit input),
restated in numpy with the reference's segment-end tables and search -- not from the device kernel's __clz form.

  μ-law  v = x >> 2 (arithmetic); v < 0: mask 0x7F, v = -v, else mask 0xFF; v = min(v, 8159) + 33;
         seg = first i with v <= SEG_UEND[i]; seg 8 (none): 0x7F ^ mask, else ((seg << 4) | ((v >> (seg + 1)) & 0xF)) ^ mask
  A-law  v = x >> 3; v >= 0: mask 0xD5, else mask 0x55, v = -v - 1;
         seg = first i with v <= SEG_AEND[i]; ((seg << 4) | ((v >> (1 if seg < 2 else seg)) & 0xF)) ^ mask
No zero-code suppression.  Packed layout of a session: utterance u at off[u], one byte per sample, the next one at
off[u] + up8(cnt[u]), the padding bytes the law's code for silence.
"""
from __future__ import annotations

import struct

import numpy as np

ULAW, ALAW = 1, 2   # CTTS_GPU_G711_ULAW, CTTS_GPU_G711_ALAW
SILENCE = {ULAW: 0xFF, ALAW: 0xD5}
SEG_UEND = np.array([0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF, 0x1FFF], np.int32)
SEG_AEND = np.array([0x1F, 0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF], np.int32)


def _search(v: np.ndarray, table: np.ndarray) -> np.ndarray:
    """The reference's search(): index of the first table entry >= v, len(table) when there is none."""
    return np.searchsorted(table, v, side="left").astype(np.int32)


def lin2ulaw(x) -> np.ndarray:
    v = np.asarray(x, np.int16).astype(np.int32) >> 2
    mask = np.where(v < 0, 0x7F, 0xFF)
    v = np.minimum(np.abs(v), 8159) + 33
    seg = _search(v, SEG_UEND)
    s = np.minimum(seg, 7)
    uval = np.where(seg >= 8, 0x7F, (s << 4) | ((v >> (s + 1)) & 0xF))
    return (uval ^ mask).astype(np.uint8)


def lin2alaw(x) -> np.ndarray:
    v = np.asarray(x, np.int16).astype(np.int32) >> 3
    mask = np.where(v >= 0, 0xD5, 0x55)
    v = np.where(v >= 0, v, -v - 1)
    seg = _search(v, SEG_AEND)
    s = np.minimum(seg, 7)
    aval = np.where(seg >= 8, 0x7F, (s << 4) | ((v >> np.where(s < 2, 1, s)) & 0xF))
    return (aval ^ mask).astype(np.uint8)


def encode(x, law: int) -> np.ndarray:
    return lin2ulaw(x) if law == ULAW else lin2alaw(x)


def table(law: int) -> np.ndarray:
    """The 65 536 codes of x = -32768 .. 32767, ascending."""
    return encode(np.arange(-32768, 32768, dtype=np.int16), law)


def up8(n: int) -> int:
    return (n + 7) // 8 * 8


def packed(pcm: list[np.ndarray], law: int) -> bytes:
    """What a G.711 session writes for utterances whose PCM session output is `pcm`: codes, silence padding to 8."""
    out = bytearray()
    for x in pcm:
        out += encode(x, law).tobytes() + bytes([SILENCE[law]]) * (up8(len(x)) - len(x))
    return bytes(out)


def parse_wav(data: bytes) -> dict:
    """A reader of the G.711 .wav files the command line writes, field by field; raises on anything else."""
    assert data[0:4] == b"RIFF" and data[8:12] == b"WAVE", "RIFF/WAVE"
    riff = struct.unpack_from("<I", data, 4)[0]
    assert riff == len(data) - 8, f"RIFF size {riff} for {len(data)} bytes"
    assert data[12:16] == b"fmt " and struct.unpack_from("<I", data, 16)[0] == 18, "fmt chunk of 18 bytes"
    tag, ch, rate, byte_rate, align, bits, cb = struct.unpack_from("<HHIIHHH", data, 20)
    assert tag in (6, 7) and ch == 1 and byte_rate == rate and align == 1 and bits == 8 and cb == 0, "fmt fields"
    assert data[38:42] == b"fact" and struct.unpack_from("<I", data, 42)[0] == 4, "fact chunk"
    frames = struct.unpack_from("<I", data, 46)[0]
    assert data[50:54] == b"data", "data chunk"
    n = struct.unpack_from("<I", data, 54)[0]
    assert n == frames, "fact and data counts"
    assert len(data) == 58 + n + (n & 1), "payload and pad byte"
    assert n % 2 == 0 or data[-1] == 0, "pad byte"
    return {"law": ULAW if tag == 7 else ALAW, "rate": rate, "count": n, "codes": np.frombuffer(data[58:58 + n], np.uint8)}
