/*
 * true_peak_oracle.c -- the CPU restatement of the true-peak ceiling of the loudness normalization
 * (ctts_gpu_set_loudness_true_peak, DESIGN.md 3.6), written from the contract alone (it shares no code with the
 * product).  The loudness L comes from tests/loudness_oracle.c; this file restates what the ceiling adds:
 *
 *   h      h[j] = sinc((j - 24) / 4) * 0.5 * (1 - cos(2 pi j / 48)), j = 0 .. 48, in double, |h[j]| <= 1e-9 set to 0,
 *          each rounded to float once
 *   P      v[m] = sum over the j with 0 <= m - 4j + 24 <= 48 of x[j] h[m - 4j + 24] (x zero outside [0, n)), for
 *          m = -24 .. 4(n - 1) + 24: ascending j, accumulator 0.0f, one fmaf per term; P = max |v[m]| as a float
 *   gain   k = clamp(floor(100 (T - L) + 0.5), -8000, 8000), table[k] = floor(65536 10^(k / 2000)),
 *          A = floor(32767 10^(C / 20)), G = min(table[k], floor((A - 1) 65536 / P)) with the division in double;
 *          65536 when L is undefined
 *   y      (x G + 32768) >> 16 in 64-bit integers (floor)
 */
#include <math.h>
#include <stdint.h>

#define ORACLE_PI 3.14159265358979323846

void ctts_oracle_true_peak_taps(float* h) {
    for (int j = 0; j <= 48; j++) {
        const double t = ((double)j - 24.0) / 4.0;
        const double sinc = t == 0.0 ? 1.0 : sin(ORACLE_PI * t) / (ORACLE_PI * t);
        const double w = 0.5 * (1.0 - cos(2.0 * ORACLE_PI * (double)j / 48.0));
        const double v = sinc * w;
        h[j] = fabs(v) <= 1e-9 ? 0.0f : (float)v;
    }
}

float ctts_oracle_true_peak(const int16_t* x, uint64_t n) {
    if (n == 0) return 0.0f;
    float h[49];
    ctts_oracle_true_peak_taps(h);
    float P = 0.0f;
    for (int64_t m = -24; m <= 4 * ((int64_t)n - 1) + 24; m++) {
        float acc = 0.0f;
        /* j from ceil((m - 24) / 4) to floor((m + 24) / 4) */
        const int64_t jlo = m - 24 >= 0 ? (m - 24 + 3) / 4 : -((24 - m) / 4);
        for (int64_t j = jlo; 4 * j <= m + 24; j++) {
            const float xj = (j >= 0 && j < (int64_t)n) ? (float)x[j] : 0.0f;
            acc = fmaf(xj, h[m - 4 * j + 24], acc);
        }
        const float a = fabsf(acc);
        if (a > P) P = a;
    }
    return P;
}

uint32_t ctts_oracle_true_peak_gain(double L, float T, float C, float P) {
    if (!(L > -INFINITY)) return 65536u;
    double k = floor(100.0 * ((double)T - L) + 0.5);
    if (k < -8000.0) k = -8000.0;
    if (k > 8000.0) k = 8000.0;
    double G = floor(65536.0 * pow(10.0, k / 2000.0));
    if (P > 0.0f) {
        const uint32_t A = (uint32_t)floor(32767.0 * pow(10.0, (double)C / 20.0));
        const double lim = floor((double)(A - 1u) * 65536.0 / (double)P);
        if (lim < G) G = lim;
    }
    return (uint32_t)G;
}

void ctts_oracle_true_peak_apply(const int16_t* x, uint64_t n, uint32_t G, int16_t* y) {
    for (uint64_t i = 0; i < n; i++) y[i] = (int16_t)(((int64_t)x[i] * (int64_t)G + 32768) >> 16);
}
