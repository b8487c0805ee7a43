// resample.cuh -- output-rate conversion (DESIGN.md 3.4): native 22 050 Hz slots -> output-rate slots.
//
// y[m] = sum_j x[j] * g[m*M + c - j*L] over 0 <= j < n, with g the Kaiser-windowed sinc of ctts_tables.c.  With
// t = m*M + c, jmax = t / L and phase phi = t - jmax*L, the taps of output m are g[phi + L*i], i = jmax - j.  The
// table is stored by phase, each row in the order the sum walks it (ascending j, i.e. descending i) and padded with
// zeros in front to a multiple of 4: row[phi][k] = g[phi + L*(kp - 1 - k)], so output m is
//   acc = 0; for k in [0, kp): acc = fmaf(x[jmax - kp + 1 + k], row[phi][k], acc)
// with x = 0 outside [0, n).  The extra terms are exact zeros and leave the float sum unchanged, so the result is
// the one of the plain ascending-j loop (tests/resample_oracle.c).
#pragma once
#include <cstdint>

namespace ctts {

constexpr int RS_THREADS = 256;
constexpr int RS_COPIES = 4;   // outputs per thread: m, m + L, m + 2L, m + 3L (one phase: every tap load serves 4 FMAs)

struct ResampleArgs {
    const int16_t* in;                  // native slots
    const unsigned long long* in_off;   // per utterance
    const uint32_t* in_counts;
    int16_t* out;                       // output-rate slots
    const unsigned long long* out_off;
    uint32_t* out_counts;
    const float4* taps;                 // L rows of kp / 4 vectors
    uint32_t L, M, kp, c;
    uint32_t smem_floats;               // staging capacity (host bound on the input span of a tile)
};

__device__ __forceinline__ int16_t rs_f2s(float v) {   // round half to even, saturate
    short r;
    asm("cvt.rni.sat.s16.f32 %0, %1;" : "=h"(r) : "f"(v));
    return (int16_t)r;
}

// Utterance blockIdx.y, tile blockIdx.x.  Work item w of an utterance stands for the outputs
// m0 + q*L (q < RS_COPIES) with m0 = (w / L) * L * RS_COPIES + w % L; a tile is RS_THREADS consecutive items.  The
// tile's input span is staged in shared memory as float (zeros outside [0, n)); then every thread walks its phase's
// row once, 4 taps per 16-byte load, for all of its outputs.
__global__ void __launch_bounds__(RS_THREADS) resample_kernel(ResampleArgs a) {
    extern __shared__ float rs_x[];
    const uint32_t u = blockIdx.y;
    const uint32_t n = a.in_counts[u];
    const uint64_t L = a.L, M = a.M;
    const uint64_t n_out = ((uint64_t)n * L + M - 1) / M;
    if (blockIdx.x == 0 && threadIdx.x == 0) a.out_counts[u] = (uint32_t)n_out;
    const uint64_t row = L * RS_COPIES;
    const uint64_t items = (n_out + row - 1) / row * L;
    const uint64_t w0 = (uint64_t)blockIdx.x * RS_THREADS;
    if (w0 >= items) return;
    const uint64_t w_last = min(items, w0 + RS_THREADS) - 1;
    auto first_out = [&](uint64_t w) { return (w / L) * row + w % L; };
    const uint64_t m_first = first_out(w0);
    // the last row's items past n_out have no output: a tile made of them alone (the items of a row are spread
    // over tiles when L > RS_THREADS) has nothing to do, and its span below would be empty
    if (m_first >= n_out) return;
    const uint64_t m_last = min(n_out - 1, first_out(w_last) + (RS_COPIES - 1) * L);
    const int64_t x_lo = (int64_t)((m_first * M + a.c) / L) - (int64_t)a.kp + 1;
    const int64_t x_hi = (int64_t)((m_last * M + a.c) / L);
    const uint32_t span = (uint32_t)(x_hi - x_lo + 1);   // <= smem_floats (host bound)

    const int16_t* src = a.in + a.in_off[u];
    for (uint32_t i = threadIdx.x; i < span; i += RS_THREADS) {
        const int64_t j = x_lo + (int64_t)i;
        rs_x[i] = (j >= 0 && j < (int64_t)n) ? (float)src[j] : 0.0f;
    }
    __syncthreads();

    const uint64_t w = w0 + threadIdx.x;
    if (w > w_last) return;
    const uint64_t m0 = first_out(w);
    if (m0 >= n_out) return;
    const uint64_t t0 = m0 * M + a.c;
    const uint64_t jmax0 = t0 / L;
    const uint32_t phi = (uint32_t)(t0 - jmax0 * L);
    // start of every output's window in the staging buffer; outputs past the end reuse the first one's
    uint32_t base[RS_COPIES];
    bool live[RS_COPIES];
#pragma unroll
    for (int q = 0; q < RS_COPIES; q++) {
        live[q] = m0 + (uint64_t)q * L < n_out;
        const int64_t jm = (int64_t)jmax0 + (live[q] ? (int64_t)q * (int64_t)M : 0);
        base[q] = (uint32_t)(jm - (int64_t)a.kp + 1 - x_lo);
    }
    const float4* tap = a.taps + (size_t)phi * (a.kp >> 2);
    float acc[RS_COPIES];
#pragma unroll
    for (int q = 0; q < RS_COPIES; q++) acc[q] = 0.0f;
    for (uint32_t k4 = 0; k4 < (a.kp >> 2); k4++) {
        const float4 g = __ldg(tap + k4);
#pragma unroll
        for (int q = 0; q < RS_COPIES; q++) {
            const float* x = rs_x + base[q] + 4u * k4;
            acc[q] = __fmaf_rn(x[0], g.x, acc[q]);
            acc[q] = __fmaf_rn(x[1], g.y, acc[q]);
            acc[q] = __fmaf_rn(x[2], g.z, acc[q]);
            acc[q] = __fmaf_rn(x[3], g.w, acc[q]);
        }
    }
    int16_t* dst = a.out + a.out_off[u];
#pragma unroll
    for (int q = 0; q < RS_COPIES; q++)
        if (live[q]) dst[m0 + (uint64_t)q * L] = rs_f2s(acc[q]);
}

}  // namespace ctts
