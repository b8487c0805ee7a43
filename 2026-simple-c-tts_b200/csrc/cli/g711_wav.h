/*
 * g711_wav.h -- the header of a G.711 .wav file (what ctts_b200 writes for g711=ulaw|alaw): 58 bytes, little endian.
 *
 *   "RIFF" <50 + count + pad> "WAVE"
 *   "fmt " <18> format tag (7 μ-law, 6 A-law), 1 channel, rate, rate bytes/s, block align 1, 8 bits, cbSize 0
 *   "fact" <4>  count                       (non-PCM WAV requires the sample count)
 *   "data" <count>                          then the count bytes and, when count is odd, one pad byte (0)
 */
#ifndef CTTS_G711_WAV_H
#define CTTS_G711_WAV_H

#include <stdint.h>

#include "ctts_gpu.h"

#define G711_WAV_HEADER_BYTES 58

static void g711_wav_put(uint8_t* p, uint32_t v, int bytes) {
    for (int i = 0; i < bytes; i++) p[i] = (uint8_t)(v >> (8 * i));
}

/* law: CTTS_GPU_G711_ULAW or CTTS_GPU_G711_ALAW; count: samples (= data bytes) */
static void g711_wav_header(uint8_t h[G711_WAV_HEADER_BYTES], int law, uint32_t rate, uint32_t count) {
    static const char tags[] = "RIFF....WAVEfmt ";
    for (int i = 0; i < 16; i++) h[i] = (uint8_t)tags[i];
    g711_wav_put(h + 4, 50u + count + (count & 1u), 4);
    g711_wav_put(h + 16, 18, 4);
    g711_wav_put(h + 20, law == CTTS_GPU_G711_ULAW ? 7 : 6, 2);
    g711_wav_put(h + 22, 1, 2);
    g711_wav_put(h + 24, rate, 4);
    g711_wav_put(h + 28, rate, 4);
    g711_wav_put(h + 32, 1, 2);
    g711_wav_put(h + 34, 8, 2);
    g711_wav_put(h + 36, 0, 2);
    h[38] = 'f'; h[39] = 'a'; h[40] = 'c'; h[41] = 't';
    g711_wav_put(h + 42, 4, 4);
    g711_wav_put(h + 46, count, 4);
    h[50] = 'd'; h[51] = 'a'; h[52] = 't'; h[53] = 'a';
    g711_wav_put(h + 54, count, 4);
}

#endif /* CTTS_G711_WAV_H */
