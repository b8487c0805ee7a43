/*
 * stretch_hop_oracle.c -- TEST INFRASTRUCTURE, not product code.
 *
 * The time_stretch loop of oracle/ctts_oracle.c after its speed -> hop step, at any synthesis hop, so that what the
 * stretch does can be examined at hops no speed reaches (127 among them).  Its offset search is the oracle's own
 * ctts_oracle_wsola_offset, passed in by the caller.  Compiled as C99 with -ffp-contract=off by
 * tests/test_wsola_pitch.py, which checks it against ctts_oracle_time_stretch at the hops a speed reaches.
 */
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define WS_FRAME 512
#define WS_HOP 128

typedef int (*wsola_offset_fn)(const int16_t* in, size_t n, const int16_t* prev_frame, size_t nominal);

static inline int16_t f2s(float v) { return (int16_t)(int32_t)v; }

static inline float clamp16f(float v) {
    if (v > 32767.0f) v = 32767.0f;
    if (v < -32768.0f) v = -32768.0f;
    return v;
}

/* room stretch_hop_oracle_stretch needs in y: frames * hop + 512 + 1024, frames = max(1, (n - 512) / 128 + 1) */
size_t stretch_hop_oracle_stretch_cap(size_t n, uint32_t hop) {
    const size_t frames = n > WS_FRAME ? (n - WS_FRAME) / WS_HOP + 1 : 1;
    return frames * hop + WS_FRAME + 1024;
}

/* y = time_stretch of in[0 .. n) at synthesis hop `hop` (frames while nominal + 512 <= n, Hann overlap-add with int16
 * wrap-around, the norm division, trailing zeros stripped).  Returns |y|, -1 when out of memory; *frames_out: frames. */
int64_t stretch_hop_oracle_stretch(wsola_offset_fn offset, const float* hann512, const int16_t* in, size_t n, uint32_t hop,
                             int16_t* y, uint32_t* frames_out) {
    const size_t cap = stretch_hop_oracle_stretch_cap(n, hop);
    float* norm = calloc(cap, sizeof *norm);
    if (!norm) return -1;
    memset(y, 0, cap * sizeof *y);
    int16_t prev[WS_FRAME];
    int have_prev = 0;
    size_t nominal = 0, syn = 0, used = 0;
    uint32_t nf = 0;
    while (nominal + WS_FRAME <= n && syn + WS_FRAME <= cap) {
        const int off = have_prev ? offset(in, n, prev, nominal) : 0;
        size_t pos = nominal + off;
        if (pos + WS_FRAME > n) pos = n - WS_FRAME;
        for (size_t i = 0; i < WS_FRAME; i++) {
            const float v = in[pos + i] * hann512[i];
            y[syn + i] = (int16_t)(y[syn + i] + f2s(v));
            norm[syn + i] += hann512[i];
            prev[i] = in[pos + i];
        }
        have_prev = 1;
        if (syn + WS_FRAME > used) used = syn + WS_FRAME;
        nominal += WS_HOP;
        syn += hop;
        nf++;
    }
    for (size_t i = 0; i < used; i++)
        if (norm[i] > 0.01f) y[i] = f2s(clamp16f(y[i] / norm[i]));
    free(norm);
    while (used > 0 && y[used - 1] == 0) used--;
    *frames_out = nf;
    return (int64_t)used;
}
