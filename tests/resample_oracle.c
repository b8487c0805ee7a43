/*
 * resample_oracle.c -- TEST INFRASTRUCTURE, not product code.
 *
 * CPU restatement of the output-rate conversion of DESIGN.md 3.4, written from the contract and not from the
 * product's code (csrc/gpu/ctts_tables.c, resample.cuh), so that the device kernel is checked against something
 * independent.  Compiled as C99 with -ffp-contract=off; tests/resample_oracle.py binds it.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdlib.h>

#define NATIVE_RATE 22050u
#define ZERO_CROSSINGS 40u

static uint32_t gcd(uint32_t a, uint32_t b) { return b ? gcd(b, a % b) : a; }

/* L / M = hz / 22050 reduced; -1 when hz is not an accepted rate */
int ctts_oracle_resample_ratio(uint32_t hz, uint32_t* L, uint32_t* M) {
    if (hz < 8000u || hz > 48000u) return -1;
    const uint32_t g = gcd(NATIVE_RATE, hz);
    *L = hz / g;
    *M = NATIVE_RATE / g;
    return (*L > 1024u || *M > 1024u) ? -1 : 0;
}

static double i0(double x) {   /* sum over k of ((x/2)^k / k!)^2 */
    double s = 0.0, t = 1.0;
    for (int k = 0; k < 1000; k++) {
        if (k > 0) t *= (x / (2.0 * k)) * (x / (2.0 * k));
        s += t;
        if (t <= s * 1e-18) break;
    }
    return s;
}

/* g[0 .. N) = float(L * firwin(N, 0.94 / R, window=('kaiser', 0.1102 * (70 - 8.7)))), N = 2 * 40 * R + 1.
 * Returns N, or 0 when hz is not accepted or cap is too small. */
size_t ctts_oracle_resample_taps(uint32_t hz, float* g, size_t cap) {
    uint32_t L, M;
    if (ctts_oracle_resample_ratio(hz, &L, &M)) return 0;
    const uint32_t R = L > M ? L : M;
    const size_t N = 2u * ZERO_CROSSINGS * R + 1u;
    if (cap < N) return 0;
    const double pi = 3.14159265358979323846, fc = 0.94 / R, beta = 0.1102 * (70.0 - 8.7);
    const double alpha = (double)(N - 1) / 2.0;
    double* h = malloc(N * sizeof *h);
    if (!h) return 0;
    double dc = 0.0;
    for (size_t i = 0; i < N; i++) {
        const double m = (double)i - alpha;
        const double ideal = m == 0.0 ? fc : sin(pi * fc * m) / (pi * m);
        const double r = m / alpha;
        const double arg = 1.0 - r * r;
        h[i] = ideal * i0(beta * sqrt(arg > 0.0 ? arg : 0.0)) / i0(beta);
        dc += h[i];
    }
    for (size_t i = 0; i < N; i++) g[i] = (float)(h[i] / dc * (double)L);
    free(h);
    return N;
}

/* ceil(n * L / M) */
uint64_t ctts_oracle_resample_count(uint32_t hz, uint64_t n) {
    uint32_t L, M;
    if (ctts_oracle_resample_ratio(hz, &L, &M)) return 0;
    return (n * L + M - 1) / M;
}

/* y[m] = sum_j x[j] g[m M + c - j L] over 0 <= j < n and 0 <= m M + c - j L < N, c = 40 R: one fmaf per term in
 * ascending j from 0.0f, then round half to even and saturate to int16.  y has room for
 * ctts_oracle_resample_count(hz, n) samples.  Returns that count, or -1 when hz is not accepted. */
int64_t ctts_oracle_resample(uint32_t hz, const int16_t* x, uint64_t n, int16_t* y) {
    uint32_t L, M;
    if (ctts_oracle_resample_ratio(hz, &L, &M)) return -1;
    const uint32_t R = L > M ? L : M;
    const size_t N = 2u * ZERO_CROSSINGS * R + 1u;
    float* g = malloc(N * sizeof *g);
    if (!g) return -1;
    ctts_oracle_resample_taps(hz, g, N);
    const uint64_t c = (uint64_t)ZERO_CROSSINGS * R, n_out = (n * L + M - 1) / M;
    for (uint64_t m = 0; m < n_out; m++) {
        const uint64_t t = m * M + c;
        const uint64_t j0 = t + 1 > N ? (t + 1 - N + L - 1) / L : 0;   /* smallest j with t - j L < N */
        uint64_t j1 = t / L;                                            /* largest j with t - j L >= 0 */
        if (j1 > n - 1) j1 = n - 1;
        float acc = 0.0f;
        for (uint64_t j = j0; j <= j1 && j < n; j++) acc = fmaf((float)x[j], g[t - j * L], acc);
        long v = lrintf(acc);
        y[m] = (int16_t)(v > 32767 ? 32767 : v < -32768 ? -32768 : v);
    }
    free(g);
    return (int64_t)n_out;
}
