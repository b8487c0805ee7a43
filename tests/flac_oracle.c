/*
 * flac_oracle.c -- the FLAC encoder contract of DESIGN.md 3.5 restated in plain C, one sample at a time, for the
 * tests.  Shares no code with the device encoder (csrc/gpu/flac.cuh) or with tests/flac_decode.c.
 *
 *   int64_t ctts_flac_oracle_encode(const int16_t* x, uint64_t n, uint32_t hz, uint8_t* out, uint64_t cap)
 *     -> the bytes of the .flac file of x, or -1 when cap is too small.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define BLOCK 4096

typedef struct {
    uint8_t* p;
    uint64_t cap, bits;   /* bits written so far */
    int overflow;
} bw;

static void put(bw* w, uint32_t len, uint64_t v) {   /* the low len bits of v, MSB first */
    while (len) {
        const uint64_t byte = w->bits >> 3;
        if (byte >= w->cap) {
            w->overflow = 1;
            return;
        }
        const uint32_t room = 8 - (uint32_t)(w->bits & 7), take = len < room ? len : room;
        if (room == 8) w->p[byte] = 0;
        w->p[byte] |= (uint8_t)(((v >> (len - take)) & ((1u << take) - 1)) << (room - take));
        w->bits += take;
        len -= take;
    }
}

static uint32_t crc8(const uint8_t* p, uint64_t n) {
    uint32_t c = 0;
    for (uint64_t i = 0; i < n; i++) {
        c ^= p[i];
        for (int b = 0; b < 8; b++) c = (c & 0x80) ? ((c << 1) ^ 0x07) & 0xff : (c << 1) & 0xff;
    }
    return c;
}

static uint32_t crc16(const uint8_t* p, uint64_t n) {
    uint32_t c = 0;
    for (uint64_t i = 0; i < n; i++) {
        c ^= (uint32_t)p[i] << 8;
        for (int b = 0; b < 8; b++) c = (c & 0x8000) ? ((c << 1) ^ 0x8005) & 0xffff : (c << 1) & 0xffff;
    }
    return c;
}

static int64_t residual(const int16_t* x, uint32_t i, uint32_t order) {
    static const int coef[5][5] = {{1}, {1, -1}, {1, -2, 1}, {1, -3, 3, -1}, {1, -4, 6, -4, 1}};
    int64_t r = 0;
    for (uint32_t j = 0; j <= order; j++) r += coef[order][j] * (int64_t)x[i - j];
    return r;
}

static uint64_t zigzag(int64_t r) { return r >= 0 ? (uint64_t)(2 * r) : (uint64_t)(-2 * r - 1); }

static uint32_t rate_code(uint32_t hz) {
    switch (hz) {
        case 8000: return 4;
        case 16000: return 5;
        case 22050: return 6;
        case 24000: return 7;
        case 32000: return 8;
        case 44100: return 9;
        case 48000: return 10;
        default: return 13;
    }
}

/* the encoder's choice for one frame of n samples */
typedef struct {
    int kind;   /* 0 CONSTANT, 1 VERBATIM, 2 FIXED */
    uint32_t order, po;
    uint32_t k[256];
    uint64_t bits;   /* subframe bits */
} choice;

static void choose(const int16_t* x, uint32_t n, choice* c) {
    memset(c, 0, sizeof *c);
    int constant = 1;
    for (uint32_t i = 1; i < n; i++)
        if (x[i] != x[0]) constant = 0;
    if (constant) {
        c->kind = 0;
        c->bits = 8 + 16;
        return;
    }
    /* 1. the fixed order: least sum of |residual| over samples 4 .. n-1, ties to the lower order; order 0 for n <= 4 */
    uint32_t order = 0;
    if (n > 4) {
        uint64_t best = 0;
        for (uint32_t o = 0; o <= 4; o++) {
            uint64_t sum = 0;
            for (uint32_t i = 4; i < n; i++) {
                const int64_t r = residual(x, i, o);
                sum += (uint64_t)(r < 0 ? -r : r);
            }
            if (o == 0 || sum < best) {
                best = sum;
                order = o;
            }
        }
    }
    /* 2. partition order and Rice parameters: fewest bits, ties to the smaller po, then the smaller k */
    uint64_t z[BLOCK];
    for (uint32_t i = order; i < n; i++) z[i] = zigzag(residual(x, i, order));
    uint64_t best_bits = UINT64_MAX;
    uint32_t best_po = 0, best_k[256];
    for (uint32_t po = 0; po <= 8 && n % (1u << po) == 0 && (n >> po) > order; po++) {
        const uint32_t P = 1u << po, m = n >> po;
        uint64_t bits = 0;
        uint32_t ks[256];
        for (uint32_t j = 0; j < P; j++) {
            const uint32_t a = j ? j * m : order, b = (j + 1) * m;
            uint64_t pb = UINT64_MAX;
            for (uint32_t k = 0; k <= 14; k++) {
                uint64_t t = (uint64_t)(b - a) * (k + 1);
                for (uint32_t i = a; i < b; i++) t += z[i] >> k;
                if (t < pb) {
                    pb = t;
                    ks[j] = k;
                }
            }
            bits += 4 + pb;
        }
        if (bits < best_bits) {
            best_bits = bits;
            best_po = po;
            memcpy(best_k, ks, sizeof ks);
        }
    }
    const uint64_t fixed = 8 + 16ull * order + 2 + 4 + best_bits, verbatim = 8 + 16ull * n;
    /* 3. VERBATIM only when strictly smaller */
    if (verbatim < fixed) {
        c->kind = 1;
        c->bits = verbatim;
        return;
    }
    c->kind = 2;
    c->order = order;
    c->po = best_po;
    memcpy(c->k, best_k, sizeof best_k);
    c->bits = fixed;
}

static void put_header(bw* w, uint32_t frame, uint32_t n, uint32_t hz) {
    const uint64_t start = w->bits >> 3;
    const uint32_t rc = rate_code(hz), bc = n == BLOCK ? 12 : (n <= 256 ? 6 : 7);
    put(w, 16, 0xfff8);
    put(w, 4, bc);
    put(w, 4, rc);
    put(w, 4, 0);   /* mono */
    put(w, 3, 4);   /* 16 bit */
    put(w, 1, 0);
    if (frame < 0x80) {
        put(w, 8, frame);
    } else {
        int extra = 1;
        while (extra < 6 && frame >= (1u << (5 * extra + 6))) extra++;
        put(w, (uint32_t)extra + 1, (1u << (extra + 1)) - 1);   /* extra + 1 one-bits, then a zero */
        put(w, 1, 0);
        put(w, 6 - (uint32_t)extra, frame >> (6 * extra));
        for (int i = extra - 1; i >= 0; i--) {
            put(w, 2, 2);
            put(w, 6, (frame >> (6 * i)) & 0x3f);
        }
    }
    if (bc == 6) put(w, 8, n - 1);
    if (bc == 7) put(w, 16, n - 1);
    if (rc == 13) put(w, 16, hz);
    if (!w->overflow) put(w, 8, crc8(w->p + start, (w->bits >> 3) - start));
}

int64_t ctts_flac_oracle_encode(const int16_t* x, uint64_t n, uint32_t hz, uint8_t* out, uint64_t cap) {
    bw w = {out, cap, 0, 0};
    const uint64_t frames = (n + BLOCK - 1) / BLOCK;
    choice* all = malloc((frames ? frames : 1) * sizeof *all);
    if (!all) return -1;
    /* STREAMINFO's frame sizes first: one pass of the choices */
    uint32_t lo = 0, hi = 0;
    for (uint64_t f = 0; f < frames; f++) {
        const uint32_t len = (uint32_t)(n - f * BLOCK < BLOCK ? n - f * BLOCK : BLOCK);
        choice* c = all + f;
        choose(x + f * BLOCK, len, c);
        uint8_t tmp[32];
        bw hw = {tmp, sizeof tmp, 0, 0};
        put_header(&hw, (uint32_t)f, len, hz);
        const uint32_t bytes = (uint32_t)((hw.bits >> 3) + (c->bits + 7) / 8 + 2);
        if (f == 0 || bytes < lo) lo = bytes;
        if (bytes > hi) hi = bytes;
    }
    put(&w, 32, 0x664c6143);   /* "fLaC" */
    put(&w, 1, 1);             /* last metadata block */
    put(&w, 7, 0);             /* STREAMINFO */
    put(&w, 24, 34);
    put(&w, 16, BLOCK);
    put(&w, 16, BLOCK);
    put(&w, 24, lo);
    put(&w, 24, hi);
    put(&w, 20, hz);
    put(&w, 3, 0);
    put(&w, 5, 15);
    put(&w, 36, n);
    for (int i = 0; i < 4; i++) put(&w, 32, 0);   /* MD5 not computed */
    for (uint64_t f = 0; f < frames && !w.overflow; f++) {
        const int16_t* s = x + f * BLOCK;
        const uint32_t len = (uint32_t)(n - f * BLOCK < BLOCK ? n - f * BLOCK : BLOCK);
        const uint64_t start = w.bits >> 3;
        const choice* c = all + f;
        put_header(&w, (uint32_t)f, len, hz);
        put(&w, 1, 0);
        if (c->kind == 0) {
            put(&w, 6, 0);
            put(&w, 1, 0);
            put(&w, 16, (uint16_t)s[0]);
        } else if (c->kind == 1) {
            put(&w, 6, 1);
            put(&w, 1, 0);
            for (uint32_t i = 0; i < len; i++) put(&w, 16, (uint16_t)s[i]);
        } else {
            put(&w, 6, 8 + c->order);
            put(&w, 1, 0);
            for (uint32_t i = 0; i < c->order; i++) put(&w, 16, (uint16_t)s[i]);
            put(&w, 2, 0);
            put(&w, 4, c->po);
            const uint32_t P = 1u << c->po, m = len >> c->po;
            for (uint32_t j = 0; j < P; j++) {
                put(&w, 4, c->k[j]);
                for (uint32_t i = j ? j * m : c->order; i < (j + 1) * m; i++) {
                    const uint64_t z = zigzag(residual(s, i, c->order));
                    for (uint64_t q = z >> c->k[j]; q > 0; q -= q < 32 ? q : 32) put(&w, q < 32 ? (uint32_t)q : 32, 0);
                    put(&w, 1, 1);
                    put(&w, c->k[j], z & ((1u << c->k[j]) - 1));
                }
            }
        }
        while (w.bits & 7) put(&w, 1, 0);
        if (!w.overflow) put(&w, 16, crc16(w.p + start, (w.bits >> 3) - start));
    }
    free(all);
    return w.overflow ? -1 : (int64_t)(w.bits >> 3);
}
