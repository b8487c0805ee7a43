/*
 * loudness_oracle.c -- the CPU restatement of the loudness normalization contract (DESIGN.md 3.6), sequential and in
 * double, written from the contract alone (it shares no code with the product):
 *
 *   x      the utterance's n output-rate int16 samples at fs Hz; the filter input is x / 32768.0
 *   K-weighting  pre-filter (high shelf) then RLB high-pass, two biquads in direct form I from zero state, with
 *          libebur128's parameterisation (shelf f0 = 1681.974450955533, G = 3.999843853973347 dB,
 *          Q = 0.7071752369554196, Vb = Vh^0.4996667741545416; high-pass f0 = 38.13547087602444,
 *          Q = 0.5003270373238773; K = tan(pi f0 / fs))
 *   blocks sub-block k = [floor(k fs / 10), floor((k + 1) fs / 10)); block j = sub-blocks j .. j + 3, complete ones
 *          only; z_j = (sum of y^2 over its samples) / (its length)
 *   gates  absolute: z_j > 10^((-70 + 0.691) / 10); relative: z_j > m / 10, m the mean of the absolute-gated z_j
 *   L      -0.691 + 10 log10(mean of the z_j that pass both); undefined (-inf) when no block passes
 *   gain   k = clamp(floor(100 (T - L) + 0.5), -8000, 8000), table[k] = floor(65536 10^(k / 2000)),
 *          A = floor(32767 10^(C / 20)), P = max |x|, G = min(table[k], floor(A 65536 / P)); 65536 when L is undefined
 *   y      (x G + 32768) >> 16 in 64-bit integers (floor)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

#define ORACLE_PI 3.14159265358979323846

void ctts_oracle_loudness_filter(uint32_t fs, double* shelf_b, double* shelf_a, double* hp_b, double* hp_a) {
    const double f0 = 1681.974450955533, G = 3.999843853973347, Q = 0.7071752369554196;
    const double K = tan(ORACLE_PI * f0 / (double)fs);
    const double Vh = pow(10.0, G / 20.0);
    const double Vb = pow(Vh, 0.4996667741545416);
    const double a0 = 1.0 + K / Q + K * K;
    shelf_b[0] = (Vh + Vb * K / Q + K * K) / a0;
    shelf_b[1] = 2.0 * (K * K - Vh) / a0;
    shelf_b[2] = (Vh - Vb * K / Q + K * K) / a0;
    shelf_a[0] = 1.0;
    shelf_a[1] = 2.0 * (K * K - 1.0) / a0;
    shelf_a[2] = (1.0 - K / Q + K * K) / a0;
    const double f1 = 38.13547087602444, Q1 = 0.5003270373238773;
    const double K1 = tan(ORACLE_PI * f1 / (double)fs);
    hp_b[0] = 1.0;
    hp_b[1] = -2.0;
    hp_b[2] = 1.0;
    hp_a[0] = 1.0;
    hp_a[1] = 2.0 * (K1 * K1 - 1.0) / (1.0 + K1 / Q1 + K1 * K1);
    hp_a[2] = (1.0 - K1 / Q1 + K1 * K1) / (1.0 + K1 / Q1 + K1 * K1);
}

static uint64_t sub_start(uint64_t k, uint32_t fs) { return k * (uint64_t)fs / 10u; }

/* integrated loudness in LUFS, -INFINITY when undefined */
double ctts_oracle_loudness(const int16_t* x, uint64_t n, uint32_t fs) {
    double sb[3], sa[3], hb[3], ha[3];
    ctts_oracle_loudness_filter(fs, sb, sa, hb, ha);
    uint64_t subs = 0;   /* complete sub-blocks */
    while (sub_start(subs + 1, fs) <= n) subs++;
    if (subs < 4) return -INFINITY;
    const uint64_t used = sub_start(subs, fs);
    double* y2 = (double*)malloc(sizeof(double) * (used ? used : 1));
    if (!y2) return NAN;
    double x1 = 0, x2 = 0, v1 = 0, v2 = 0, w1 = 0, w2 = 0;   /* direct form I histories of both stages */
    for (uint64_t i = 0; i < used; i++) {
        const double in = (double)x[i] / 32768.0;
        const double v = sb[0] * in + sb[1] * x1 + sb[2] * x2 - sa[1] * v1 - sa[2] * v2;
        x2 = x1;
        x1 = in;
        const double w = hb[0] * v + hb[1] * v1 + hb[2] * v2 - ha[1] * w1 - ha[2] * w2;
        v2 = v1;
        v1 = v;
        w2 = w1;
        w1 = w;
        y2[i] = w * w;
    }
    const uint64_t blocks = subs - 3;
    double* z = (double*)malloc(sizeof(double) * blocks);
    if (!z) { free(y2); return NAN; }
    for (uint64_t j = 0; j < blocks; j++) {
        const uint64_t b = sub_start(j, fs), e = sub_start(j + 4, fs);
        double s = 0.0;
        for (uint64_t i = b; i < e; i++) s += y2[i];
        z[j] = s / (double)(e - b);
    }
    free(y2);
    const double gate_abs = pow(10.0, (-70.0 + 0.691) / 10.0);
    double s1 = 0.0;
    uint64_t m1 = 0;
    for (uint64_t j = 0; j < blocks; j++)
        if (z[j] > gate_abs) { s1 += z[j]; m1++; }
    double L = -INFINITY;
    if (m1) {
        const double gate_rel = s1 / (double)m1 / 10.0;
        double s2 = 0.0;
        uint64_t m2 = 0;
        for (uint64_t j = 0; j < blocks; j++)
            if (z[j] > gate_abs && z[j] > gate_rel) { s2 += z[j]; m2++; }
        if (m2) L = -0.691 + 10.0 * log10(s2 / (double)m2);
    }
    free(z);
    return L;
}

uint32_t ctts_oracle_loudness_table(int k) { return (uint32_t)floor(65536.0 * pow(10.0, (double)k / 2000.0)); }

uint32_t ctts_oracle_loudness_ceiling(float C) { return (uint32_t)floor(32767.0 * pow(10.0, (double)C / 20.0)); }

uint32_t ctts_oracle_loudness_gain(double L, float T, float C, uint32_t peak) {
    if (!(L > -INFINITY)) return 65536u;
    double k = floor(100.0 * ((double)T - L) + 0.5);
    if (k < -8000.0) k = -8000.0;
    if (k > 8000.0) k = 8000.0;
    uint64_t G = ctts_oracle_loudness_table((int)k);
    if (peak) {
        const uint64_t lim = (uint64_t)ctts_oracle_loudness_ceiling(C) * 65536u / peak;
        if (lim < G) G = lim;
    }
    return (uint32_t)G;
}

/* The whole stage on one utterance: y (n samples) from x; returns G, *L receives the loudness. */
uint32_t ctts_oracle_loudness_normalize(const int16_t* x, uint64_t n, uint32_t fs, float T, float C, int16_t* y, double* L) {
    uint32_t peak = 0;
    for (uint64_t i = 0; i < n; i++) {
        const uint32_t a = (uint32_t)abs((int)x[i]);
        if (a > peak) peak = a;
    }
    *L = ctts_oracle_loudness(x, n, fs);
    const uint32_t G = ctts_oracle_loudness_gain(*L, T, C, peak);
    for (uint64_t i = 0; i < n; i++) y[i] = (int16_t)(((int64_t)x[i] * (int64_t)G + 32768) >> 16);
    return G;
}
