/*
 * ctts_tables.c -- host-computed lookup tables uploaded by ctts_gpu_init.
 *
 * Compiled as C99 with -ffp-contract=off (not by nvcc) on purpose: the
 * reference fills these tables with glibc cosf/sinf under C promotion rules
 * (PI is a double literal, ctts.c:45), and CUDA's cosf is not bit-identical to
 * libm's.  Bit-exact PCM needs bit-exact tables, so they are produced here the
 * way ctts.c:60-73 (fade LUTs), :2198-2204 (256-sample Hann) and :1624
 * (512-sample WSOLA Hann) produce them.
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>

#define CTTS_PI 3.14159265358979323846

void ctts_host_tables(float* fade_out, float* fade_in, float* sine, float* hann256, float* hann512) {
    for (int i = 0; i < 1024; i++) {
        float t = (float)i / (float)(1024 - 1);
        fade_out[i] = 0.5f * (1.0f + cosf(CTTS_PI * t));
        fade_in[i] = 0.5f * (1.0f - cosf(CTTS_PI * t));
        sine[i] = sinf(t * CTTS_PI * 0.5f);
    }
    for (int i = 0; i < 256; i++) hann256[i] = 0.5f * (1.0f - cosf(2.0f * CTTS_PI * i / 256));
    for (size_t i = 0; i < 512; i++)
        hann512[i] = 0.5f * (1.0f - cosf(2.0f * (float)CTTS_PI * (float)i / (float)512));
}

/* I0, the modified Bessel function of order 0, by its power series sum_k ((x/2)^k / k!)^2 */
static double bessel_i0(double x) {
    double term = 1.0, sum = 1.0;
    const double q = 0.25 * x * x;
    for (int k = 1; k < 500; k++) {
        term *= q / ((double)k * (double)k);
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

/* The output-rate filter of DESIGN.md 3.4: g = L * firwin(N, 0.94 / R, window=('kaiser', beta)), N = 2*H*R + 1,
 * H = 40, beta = 0.1102 * (70 - 8.7), computed in double and rounded to float once.  g receives N taps. */
void ctts_host_resample_taps(unsigned L, unsigned M, float* g) {
    const unsigned R = L > M ? L : M;
    const unsigned N = 2u * 40u * R + 1u;
    const double cutoff = 0.94 / (double)R, beta = 0.1102 * (70.0 - 8.7), half = 0.5 * (double)(N - 1);
    const double i0b = bessel_i0(beta);
    double* h = (double*)malloc(sizeof(double) * N);
    double sum = 0.0;
    if (!h) return;
    for (unsigned i = 0; i < N; i++) {
        const double m = (double)i - half;
        const double a = CTTS_PI * cutoff * m;
        const double sinc = m == 0.0 ? 1.0 : sin(a) / a;
        const double r = m / half;
        const double w = bessel_i0(beta * sqrt(r * r < 1.0 ? 1.0 - r * r : 0.0)) / i0b;
        h[i] = cutoff * sinc * w;
        sum += h[i];
    }
    for (unsigned i = 0; i < N; i++) g[i] = (float)((double)L * (h[i] / sum));
    free(h);
}

/* K-weighting of ITU-R BS.1770-4 at fs Hz (DESIGN.md 3.6), in libebur128's parameterisation.  shelf receives the
 * pre-filter (high shelf) b0, b1, b2, a1, a2; hp receives a1, a2 of the RLB high-pass, whose numerator is 1, -2, 1.
 * At 48 kHz these are the two tables of BS.1770-4. */
void ctts_host_loudness_filter(unsigned fs, double* shelf, double* hp) {
    double f0 = 1681.974450955533, Q = 0.7071752369554196, K = tan(CTTS_PI * f0 / (double)fs);
    const double G = 3.999843853973347, Vh = pow(10.0, G / 20.0), Vb = pow(Vh, 0.4996667741545416);
    const double a0 = 1.0 + K / Q + K * K;
    shelf[0] = (Vh + Vb * K / Q + K * K) / a0;
    shelf[1] = 2.0 * (K * K - Vh) / a0;
    shelf[2] = (Vh - Vb * K / Q + K * K) / a0;
    shelf[3] = 2.0 * (K * K - 1.0) / a0;
    shelf[4] = (1.0 - K / Q + K * K) / a0;
    f0 = 38.13547087602444;
    Q = 0.5003270373238773;
    K = tan(CTTS_PI * f0 / (double)fs);
    hp[0] = 2.0 * (K * K - 1.0) / (1.0 + K / Q + K * K);
    hp[1] = (1.0 - K / Q + K * K) / (1.0 + K / Q + K * K);
}

/* The loudness gains in Q16, steps of 0.01 dB: table[k + 8000] = floor(65536 * 10^(k / 2000)), k = -8000 .. 8000. */
void ctts_host_loudness_gains(unsigned* table) {
    for (int k = -8000; k <= 8000; k++) table[k + 8000] = (unsigned)floor(65536.0 * pow(10.0, (double)k / 2000.0));
}

/* The sample-peak ceiling of C dBFS as an int16 magnitude: floor(32767 * 10^(C / 20)). */
unsigned ctts_host_loudness_ceiling(float ceiling_dbfs) {
    return (unsigned)floor(32767.0 * pow(10.0, (double)ceiling_dbfs / 20.0));
}

/* The true-peak interpolator (DESIGN.md 3.6): 4x oversampling, 49 taps, the windowed sinc libebur128 uses below
 * 96 kHz.  h[j] = sinc((j - 24) / 4) * 0.5 * (1 - cos(2 pi j / 48)), j = 0 .. 48, in double; |h[j]| <= 1e-9 becomes
 * exactly 0 (the non-centre taps of phase 0, so phase j mod 4 = 0 is the identity); each tap is rounded to float once. */
void ctts_host_true_peak_taps(float* h) {
    for (int j = 0; j <= 48; j++) {
        const double t = (double)(j - 24) / 4.0;
        const double s = j == 24 ? 1.0 : sin(CTTS_PI * t) / (CTTS_PI * t);
        const double v = s * 0.5 * (1.0 - cos(2.0 * CTTS_PI * (double)j / 48.0));
        h[j] = fabs(v) <= 1e-9 ? 0.0f : (float)v;
    }
}
