/*
 * flac_decode.c -- a FLAC decoder written from RFC 9639 for the tests, independent of the encoders (the device's in
 * csrc/gpu/flac.cuh and tests/flac_oracle.c).  It decodes more than the project's encoder emits -- CONSTANT,
 * VERBATIM, FIXED and LPC subframes, Rice methods 0 and 1 with the escape code, wasted bits, any blocksize and
 * sample-rate code, fixed and variable blocking -- for mono streams of 4 to 16 bits, and it rejects anything
 * malformed: a bad marker, STREAMINFO, sync code, reserved bit, CRC-8, CRC-16, frame number, or a stream whose
 * samples disagree with STREAMINFO.
 *
 *   int64_t ctts_flac_decode(const uint8_t* in, uint64_t len, int16_t* out, uint64_t cap, uint64_t* info)
 *     -> samples decoded (< 0: an error code below).  info (may be NULL) receives 9 values: min and max blocksize,
 *        min and max frame size, sample rate, channels, bits per sample, total samples, 1 if the MD5 is all zero.
 *
 *   int64_t ctts_flac_decode_report(..., uint32_t* rep, uint64_t rep_cap, uint64_t* frames)
 *     -> the same, and for every frame (at most rep_cap) what was parsed, REPORT_FIELDS values: the coded frame
 *        number, the blocksize, the header length in bytes (CRC-8 included), the subframe kind (0 CONSTANT,
 *        1 VERBATIM, 2 FIXED, 3 LPC), the predictor order, the partition order, the least and the largest Rice
 *        parameter (15: the escape code; 0 for CONSTANT and VERBATIM).  *frames receives the frames decoded.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { REPORT_FIELDS = 8, K_NONE = 255 };

typedef struct {   /* what one frame's subframe and residual said */
    uint32_t kind, order, po, kmin, kmax;
} parsed;

enum {
    E_MARKER = -1, E_METADATA = -2, E_SYNC = -3, E_RESERVED = -4, E_CRC8 = -5, E_CRC16 = -6, E_SUBFRAME = -7,
    E_RESIDUAL = -8, E_TRUNCATED = -9, E_CAPACITY = -10, E_STREAMINFO = -11, E_UNSUPPORTED = -12, E_FRAMENUM = -13,
};

typedef struct {
    const uint8_t* p;
    uint64_t len, pos;   /* pos in bits */
    int err;
} br;

static uint64_t rd(br* b, uint32_t n) {
    uint64_t v = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (b->pos >= 8 * b->len) {
            b->err = E_TRUNCATED;
            return 0;
        }
        v = (v << 1) | ((b->p[b->pos >> 3] >> (7 - (b->pos & 7))) & 1);
        b->pos++;
    }
    return v;
}

static int64_t rd_signed(br* b, uint32_t n) {
    if (n == 0) return 0;
    const uint64_t v = rd(b, n);
    return (v >> (n - 1)) & 1 ? (int64_t)v - ((int64_t)1 << n) : (int64_t)v;
}

static uint64_t rd_unary(br* b) {   /* zeros ended by a one */
    uint64_t q = 0;
    while (!b->err && rd(b, 1) == 0) q++;
    return q;
}

static uint8_t crc8_of(const uint8_t* p, uint64_t n) {
    uint8_t c = 0;
    while (n--) {
        c ^= *p++;
        for (int i = 0; i < 8; i++) c = (uint8_t)(c & 0x80 ? (c << 1) ^ 0x07 : c << 1);
    }
    return c;
}

static uint16_t crc16_of(const uint8_t* p, uint64_t n) {
    uint16_t c = 0;
    while (n--) {
        c ^= (uint16_t)(*p++ << 8);
        for (int i = 0; i < 8; i++) c = (uint16_t)(c & 0x8000 ? (c << 1) ^ 0x8005 : c << 1);
    }
    return c;
}

static int residual(br* b, uint32_t bs, uint32_t order, int64_t* r, parsed* rp) {
    const uint32_t method = (uint32_t)rd(b, 2);
    if (method > 1) return E_RESIDUAL;
    const uint32_t pbits = method ? 5 : 4, esc = method ? 31 : 15;
    const uint32_t po = (uint32_t)rd(b, 4);
    const uint32_t P = 1u << po;
    if (bs % P || (bs >> po) < order) return E_RESIDUAL;
    rp->po = po;
    uint32_t i = order;
    for (uint32_t j = 0; j < P && !b->err; j++) {
        const uint32_t end = (j + 1) * (bs >> po);
        const uint32_t k = (uint32_t)rd(b, pbits);
        if (k < rp->kmin) rp->kmin = k;
        if (k > rp->kmax) rp->kmax = k;
        if (k == esc) {
            const uint32_t w = (uint32_t)rd(b, 5);
            for (; i < end && !b->err; i++) r[i] = rd_signed(b, w);
        } else {
            for (; i < end && !b->err; i++) {
                const uint64_t q = rd_unary(b);
                const uint64_t u = (q << k) | rd(b, k);
                r[i] = (u & 1) ? -(int64_t)(u >> 1) - 1 : (int64_t)(u >> 1);
            }
        }
    }
    return b->err;
}

static int subframe(br* b, uint32_t bs, uint32_t bps, int64_t* s, int64_t* r, parsed* rp) {
    if (rd(b, 1) != 0) return E_RESERVED;
    const uint32_t type = (uint32_t)rd(b, 6);
    *rp = (parsed){type >= 32 ? 3 : type >= 8 ? 2 : type, type >= 32 ? type - 31 : type >= 8 ? type - 8 : 0, 0, K_NONE, 0};
    uint32_t wasted = 0;
    if (rd(b, 1)) wasted = (uint32_t)rd_unary(b) + 1;
    if (wasted >= bps) return E_SUBFRAME;
    const uint32_t w = bps - wasted;
    if (type == 0) {
        const int64_t v = rd_signed(b, w);
        for (uint32_t i = 0; i < bs; i++) s[i] = v;
    } else if (type == 1) {
        for (uint32_t i = 0; i < bs; i++) s[i] = rd_signed(b, w);
    } else if (type >= 8 && type <= 12) {
        static const int64_t coef[5][4] = {{0}, {1}, {2, -1}, {3, -3, 1}, {4, -6, 4, -1}};
        const uint32_t order = type - 8;
        if (order > bs) return E_SUBFRAME;
        for (uint32_t i = 0; i < order; i++) s[i] = rd_signed(b, w);
        int rc = residual(b, bs, order, r, rp);
        if (rc) return rc;
        for (uint32_t i = order; i < bs; i++) {
            int64_t p = 0;
            for (uint32_t j = 0; j < order; j++) p += coef[order][j] * s[i - 1 - j];
            s[i] = p + r[i];
        }
    } else if (type >= 32) {
        const uint32_t order = type - 31;
        if (order > bs) return E_SUBFRAME;
        for (uint32_t i = 0; i < order; i++) s[i] = rd_signed(b, w);
        const uint32_t prec = (uint32_t)rd(b, 4) + 1;
        if (prec == 16) return E_SUBFRAME;
        const int64_t shift = rd_signed(b, 5);
        if (shift < 0) return E_SUBFRAME;
        int64_t c[32];
        for (uint32_t j = 0; j < order; j++) c[j] = rd_signed(b, prec);
        int rc = residual(b, bs, order, r, rp);
        if (rc) return rc;
        for (uint32_t i = order; i < bs; i++) {
            int64_t p = 0;
            for (uint32_t j = 0; j < order; j++) p += c[j] * s[i - 1 - j];
            s[i] = (p >> shift) + r[i];
        }
    } else {
        return E_SUBFRAME;
    }
    for (uint32_t i = 0; i < bs; i++) s[i] = (int64_t)((uint64_t)s[i] << wasted);
    return b->err;
}

static int64_t decode(const uint8_t* in, uint64_t len, int16_t* out, uint64_t cap, uint64_t* info, int64_t* s, int64_t* r,
                      uint32_t* rep, uint64_t rep_cap, uint64_t* frames) {
    br b = {in, len, 0, 0};
    if (len < 4 || memcmp(in, "fLaC", 4) != 0) return E_MARKER;
    b.pos = 32;
    /* metadata: STREAMINFO first, any further blocks skipped */
    uint32_t min_bs = 0, max_bs = 0, min_fs = 0, max_fs = 0, rate = 0, ch = 0, bps = 0;
    uint64_t total = 0;
    int md5_zero = 1, last = 0, first = 1;
    while (!last) {
        last = (int)rd(&b, 1);
        const uint32_t type = (uint32_t)rd(&b, 7), blen = (uint32_t)rd(&b, 24);
        if (b.err) return E_METADATA;
        if (first != (type == 0)) return E_METADATA;
        if (type == 127) return E_METADATA;
        if (type == 0) {
            if (blen != 34) return E_METADATA;
            min_bs = (uint32_t)rd(&b, 16);
            max_bs = (uint32_t)rd(&b, 16);
            min_fs = (uint32_t)rd(&b, 24);
            max_fs = (uint32_t)rd(&b, 24);
            rate = (uint32_t)rd(&b, 20);
            ch = (uint32_t)rd(&b, 3) + 1;
            bps = (uint32_t)rd(&b, 5) + 1;
            total = rd(&b, 36);
            for (int i = 0; i < 16; i++) md5_zero &= rd(&b, 8) == 0;
            if (b.err) return E_METADATA;
            if (min_bs < 16 || max_bs < min_bs || (min_fs && max_fs && max_fs < min_fs)) return E_STREAMINFO;
        } else {
            b.pos += 8ull * blen;
            if (b.pos > 8 * len) return E_METADATA;
        }
        first = 0;
    }
    if (info) {
        const uint64_t v[9] = {min_bs, max_bs, min_fs, max_fs, rate, ch, bps, total, (uint64_t)md5_zero};
        memcpy(info, v, sizeof v);
    }
    if (ch != 1) return E_UNSUPPORTED;
    if (bps < 4 || bps > 16) return E_UNSUPPORTED;
    uint64_t done = 0, frame_no = 0;
    while (b.pos < 8 * len) {
        const uint64_t start = b.pos >> 3;
        if (b.pos & 7) return E_SYNC;
        if (rd(&b, 15) != 0x7ffc) return E_SYNC;
        const uint32_t variable = (uint32_t)rd(&b, 1);
        const uint32_t bc = (uint32_t)rd(&b, 4), rc = (uint32_t)rd(&b, 4);
        const uint32_t ca = (uint32_t)rd(&b, 4), sc = (uint32_t)rd(&b, 3);
        if (rd(&b, 1) != 0) return E_RESERVED;
        /* the coded number: UTF-8-like, up to 7 bytes */
        uint64_t num = rd(&b, 8);
        int extra = 0;
        if (num >= 0x80) {
            if (num >= 0xfe) return E_FRAMENUM;
            while (num & (0x80u >> (extra + 1))) extra++;
            if (extra == 0) return E_FRAMENUM;
            num &= 0x3fu >> extra;
            for (int i = 0; i < extra; i++) {
                const uint64_t c = rd(&b, 8);
                if ((c & 0xc0) != 0x80) return E_FRAMENUM;
                num = num << 6 | (c & 0x3f);
            }
        }
        uint32_t bs;
        if (bc == 0) return E_RESERVED;
        else if (bc == 1) bs = 192;
        else if (bc <= 5) bs = 576u << (bc - 2);
        else if (bc == 6) bs = (uint32_t)rd(&b, 8) + 1;
        else if (bc == 7) bs = (uint32_t)rd(&b, 16) + 1;
        else bs = 256u << (bc - 8);
        static const uint32_t rates[12] = {0, 88200, 176400, 192000, 8000, 16000, 22050, 24000, 32000, 44100, 48000, 96000};
        uint32_t hz;
        if (rc == 15) return E_RESERVED;
        else if (rc < 12) hz = rc ? rates[rc] : rate;
        else if (rc == 12) hz = (uint32_t)rd(&b, 8) * 1000;
        else if (rc == 13) hz = (uint32_t)rd(&b, 16);
        else hz = (uint32_t)rd(&b, 16) * 10;
        if (b.err) return b.err;
        const uint8_t crc8 = (uint8_t)rd(&b, 8);
        if (b.err) return b.err;
        if (crc8 != crc8_of(in + start, (b.pos >> 3) - start - 1)) return E_CRC8;
        if (hz != rate) return E_STREAMINFO;
        if (ca != 0) return E_UNSUPPORTED;
        static const uint32_t sizes[8] = {0, 8, 12, 0, 16, 20, 24, 32};
        if (sc == 3) return E_RESERVED;
        const uint32_t fbps = sc ? sizes[sc] : bps;
        if (fbps != bps) return E_STREAMINFO;
        if (variable ? num != done : num != frame_no) return E_FRAMENUM;
        if (bs > max_bs) return E_STREAMINFO;
        const uint64_t hdr = (b.pos >> 3) - start;
        parsed p;
        int e = subframe(&b, bs, bps, s, r, &p);
        if (e) return e;
        if (rep && frame_no < rep_cap) {
            const uint32_t v[REPORT_FIELDS] = {(uint32_t)num, bs, (uint32_t)hdr, p.kind, p.order, p.po,
                                               p.kmin == K_NONE ? 0 : p.kmin, p.kmax};
            memcpy(rep + REPORT_FIELDS * frame_no, v, sizeof v);
        }
        b.pos = (b.pos + 7) & ~7ull;
        const uint64_t crc16 = rd(&b, 16);
        if (b.err) return b.err;
        if (crc16 != crc16_of(in + start, (b.pos >> 3) - start - 2)) return E_CRC16;
        const uint64_t fs = (b.pos >> 3) - start;
        if ((min_fs && fs < min_fs) || (max_fs && fs > max_fs)) return E_STREAMINFO;
        if (done + bs > cap) return E_CAPACITY;
        for (uint32_t i = 0; i < bs; i++) {
            if (s[i] < -(1ll << (bps - 1)) || s[i] >= (1ll << (bps - 1))) return E_SUBFRAME;
            out[done + i] = (int16_t)s[i];
        }
        done += bs;
        frame_no++;
    }
    if (total && done != total) return E_STREAMINFO;
    if (frames) *frames = frame_no;
    return (int64_t)done;
}

int64_t ctts_flac_decode_report(const uint8_t* in, uint64_t len, int16_t* out, uint64_t cap, uint64_t* info, uint32_t* rep,
                                uint64_t rep_cap, uint64_t* frames) {
    int64_t* s = malloc(65536 * sizeof *s);   /* the largest blocksize */
    int64_t* r = malloc(65536 * sizeof *r);
    const int64_t rc = s && r ? decode(in, len, out, cap, info, s, r, rep, rep_cap, frames) : E_CAPACITY;
    free(s);
    free(r);
    return rc;
}

int64_t ctts_flac_decode(const uint8_t* in, uint64_t len, int16_t* out, uint64_t cap, uint64_t* info) {
    return ctts_flac_decode_report(in, len, out, cap, info, NULL, 0, NULL);
}
