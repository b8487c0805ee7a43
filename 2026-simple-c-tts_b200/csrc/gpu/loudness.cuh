// loudness.cuh -- loudness normalization of every utterance (DESIGN.md 3.6): integrated loudness after
// ITU-R BS.1770-4 (K-weighting, 400 ms blocks, absolute and relative gates), one Q16 gain per utterance that reaches
// the target without the sample peak (or, under a true-peak setting, the 4x oversampled peak of BS.1770-4 Annex 2)
// exceeding the ceiling, applied in place on the output-rate slots.
//
// The K-weighting is an IIR cascade in double, sequential by nature.  It is cut into chunks, one per 100 ms
// sub-block k = [floor(k*fs/10), floor((k+1)*fs/10)) (the last one clipped at the count):
//   ld_chunk_kernel<false>  every chunk from zero state: its end state e_k and its peak
//   ld_scan_kernel          per utterance, the true start state of every chunk: s_{k+1} = A^len_k s_k + e_k, with the
//                           zero-input transitions A^lo, A^(lo+1) of the two sub-block lengths tabulated on the host
//   ld_chunk_kernel<true>   every chunk again from its true state: sum of y^2
//   ld_true_peak_kernel     true-peak plans only: max |v| of the 4x oversampled signal per tile of 2048 positions
//   ld_gain_kernel          per utterance: block energies, both gates, L, the gain
//   ld_apply_kernel         y = (x * G + 32768) >> 16 in place, skipped where G is unity
// The filter state of a chunk is not its exact sequential value (the scan reassociates the recurrence), so L agrees
// with the sequential restatement (tests/loudness_oracle.c) to about 1e-12 relative, not bit for bit.
#pragma once
#include <cstdint>

#include "block_prims.cuh"

namespace ctts {

constexpr int LD_THREADS = 128;        // chunk passes: one chunk per thread
constexpr int LD_WARPS = LD_THREADS / 32;
constexpr int LD_SCAN_THREADS = 128;   // one utterance per thread
constexpr int LD_SCAN_BATCH = 8;       // chunk end states loaded ahead of the scan's serial chain
constexpr int LD_GAIN_THREADS = 256;   // one CTA per utterance
constexpr int LD_APPLY_THREADS = 256;
constexpr uint32_t LD_APPLY_TILE = 8u * LD_APPLY_THREADS * 4u;
constexpr int LD_TP_THREADS = 256;
constexpr int LD_TP_PER = 8;           // consecutive positions per thread, from one register window
constexpr uint32_t LD_TP_TILE = LD_TP_THREADS * LD_TP_PER;
constexpr int LD_TP_HALO = 6;          // samples staged on each side of a tile
constexpr uint32_t LD_TP_STAGE = LD_TP_TILE + 2 * LD_TP_HALO;
constexpr int LD_K_MAX = 8000;         // gain table: k = -LD_K_MAX .. LD_K_MAX hundredths of a dB
constexpr uint32_t LD_UNITY = 65536;   // G = 1 in Q16: y == x

// The K-weighting at one rate, passed by value to every kernel.  State (s1, s2, t1, t2): the transposed direct form II
// states of the pre-filter and of the RLB high-pass.
struct LdFilter {
    double b0, b1, b2;   // pre-filter numerator / 32768 (the input is x / 32768, a power of two: exact)
    double a1, a2;       // pre-filter denominator
    double h1, h2;       // RLB high-pass denominator (numerator 1, -2, 1)
    double pw[2][16];    // state transition over lo and lo + 1 samples of zero input, row major
    uint32_t fs;
    uint32_t lo;         // floor(fs / 10): every complete sub-block is lo or lo + 1 samples long
};

struct LdState {
    double s1, s2, t1, t2;
};

// One sample of the cascade (also run on the host, with x = 0, to tabulate LdFilter::pw).
__host__ __device__ __forceinline__ double ld_step(const LdFilter& f, LdState& s, double x) {
    const double y1 = fma(f.b0, x, s.s1);
    s.s1 = fma(-f.a1, y1, fma(f.b1, x, s.s2));
    s.s2 = fma(-f.a2, y1, f.b2 * x);
    const double y = y1 + s.t1;
    s.t1 = fma(-f.h1, y, fma(-2.0, y1, s.t2));
    s.t2 = fma(-f.h2, y, y1);
    return y;
}

struct LdArgs {
    int16_t* pcm;                     // output-rate slots, scaled in place by ld_apply_kernel
    const unsigned long long* off;    // slot offsets [n + 1], then the first chunk of every utterance [n + 1]
                                      // (true peak: then its first ld_true_peak_kernel tile [n + 1])
    const uint32_t* counts;           // output-rate counts
    double* state;                    // 4 per chunk: zero-state end state, overwritten by the scan with the start state
    double* energy;                   // per chunk: sum of y^2
    uint32_t* peak;                   // per chunk: max |x|
    double* lufs;                     // per utterance: L, -inf when undefined
    uint32_t* gain;                   // per utterance: G (Q16)
    const uint32_t* table;            // floor(65536 * 10^(k / 2000)) at k + LD_K_MAX
    double gate_abs;                  // 10^((-70 + 0.691) / 10)
    uint32_t n;                       // utterances of the plan
    uint32_t u0;                      // first utterance of this launch (grid.y split)
    uint32_t ceiling;                 // A = floor(32767 * 10^(C / 20))
    float target;                     // T, LUFS
    LdFilter f;
    // true-peak plans only (the fields above keep their offsets, so the sample-peak kernels are unchanged)
    float* tp_tile;                   // per (utterance, tile): max |v| over the tile's positions
    float* tp_peak;                   // per utterance: P
    float tp_h[3][12];                // phases r = 1 .. 3: tp_h[r - 1][i] = h[44 - 4i + r], the tap of x[q - 5 + i]
};

__device__ __forceinline__ unsigned long long ld_sub_start(unsigned long long k, uint32_t fs) { return k * fs / 10u; }

// Chunks of an utterance: the sub-blocks that start before its count, never more than the plan laid out for it.
__device__ __forceinline__ unsigned long long ld_chunks(const LdArgs& a, uint32_t u, uint32_t cnt) {
    const unsigned long long k = ((unsigned long long)cnt * 10u + a.f.fs - 1u) / a.f.fs;
    return min(k, a.off[a.n + 1 + u + 1] - a.off[a.n + 1 + u]);
}

struct LdSumD {
    __device__ __forceinline__ double operator()(double x, double y) const { return x + y; }
};
struct LdMaxU {
    __device__ __forceinline__ unsigned operator()(unsigned x, unsigned y) const { return x > y ? x : y; }
};

// Utterance u0 + blockIdx.y, chunks blockIdx.x * LD_THREADS + threadIdx.x.  A warp's 32 chunks lie about fs / 10
// samples apart, so the warp stages them through shared memory 32 samples at a time: one coalesced 64-byte load per
// chunk, then every thread filters its own row.
template <bool ENERGY>
__global__ void __launch_bounds__(LD_THREADS) ld_chunk_kernel(LdArgs a) {
    __shared__ int32_t stage[LD_WARPS][32][33];
    __shared__ unsigned long long wbeg[LD_WARPS][32];
    __shared__ uint32_t wlen[LD_WARPS][32];
    const uint32_t u = a.u0 + blockIdx.y;
    const uint32_t cnt = a.counts[u];
    const unsigned long long nch = ld_chunks(a, u, cnt);
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const unsigned long long k = (unsigned long long)blockIdx.x * LD_THREADS + threadIdx.x;
    if (k - lane >= nch) return;   // the whole warp
    const bool mine = k < nch;
    const unsigned long long b = ld_sub_start(k, a.f.fs);
    const uint32_t len = mine ? (uint32_t)(min(ld_sub_start(k + 1, a.f.fs), (unsigned long long)cnt) - b) : 0u;
    wbeg[w][lane] = b;
    wlen[w][lane] = len;
    const uint32_t maxlen = __reduce_max_sync(0xffffffffu, len);
    const int16_t* x = a.pcm + a.off[u];
    const unsigned long long c = a.off[a.n + 1 + u] + k;
    LdState s{0.0, 0.0, 0.0, 0.0};
    if (ENERGY && mine) {
        const double2* p = reinterpret_cast<const double2*>(a.state + 4 * c);
        const double2 q0 = p[0], q1 = p[1];
        s = LdState{q0.x, q0.y, q1.x, q1.y};
    }
    double acc = 0.0;
    uint32_t pk = 0;
    __syncwarp();
    for (uint32_t t0 = 0; t0 < maxlen; t0 += 32u) {
        const uint32_t i = t0 + lane;
#pragma unroll 8
        for (int j = 0; j < 32; j++) stage[w][j][lane] = i < wlen[w][j] ? x[wbeg[w][j] + i] : 0;
        __syncwarp();
        const uint32_t m = len > t0 ? min(32u, len - t0) : 0u;
        for (uint32_t q = 0; q < m; q++) {
            const int32_t v = stage[w][lane][q];
            const double y = ld_step(a.f, s, (double)v);
            if (ENERGY) acc = fma(y, y, acc);
            else pk = max(pk, (uint32_t)abs(v));
        }
        __syncwarp();
    }
    if (!mine) return;
    if (ENERGY) {
        a.energy[c] = acc;
    } else {
        double2* p = reinterpret_cast<double2*>(a.state + 4 * c);
        p[0] = make_double2(s.s1, s.s2);
        p[1] = make_double2(s.t1, s.t2);
        a.peak[c] = pk;
    }
}

// One utterance per thread: the chunks' end states e_k become their start states s_k in place.  Only a complete
// sub-block is followed by another chunk, so every transition is A^lo or A^(lo+1).
__global__ void __launch_bounds__(LD_SCAN_THREADS) ld_scan_kernel(LdArgs a) {
    const uint32_t u = blockIdx.x * LD_SCAN_THREADS + threadIdx.x;
    if (u >= a.n) return;
    const unsigned long long nch = ld_chunks(a, u, a.counts[u]);
    double2* st = reinterpret_cast<double2*>(a.state + 4 * a.off[a.n + 1 + u]);
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (unsigned long long k0 = 0; k0 < nch; k0 += LD_SCAN_BATCH) {
        double2 e[LD_SCAN_BATCH][2];
#pragma unroll
        for (int i = 0; i < LD_SCAN_BATCH; i++)
            if (k0 + i < nch) {
                e[i][0] = st[2 * (k0 + i)];
                e[i][1] = st[2 * (k0 + i) + 1];
            }
#pragma unroll
        for (int i = 0; i < LD_SCAN_BATCH; i++) {
            const unsigned long long k = k0 + i;
            if (k >= nch) break;
            st[2 * k] = make_double2(s[0], s[1]);
            st[2 * k + 1] = make_double2(s[2], s[3]);
            const double* P = a.f.pw[ld_sub_start(k + 1, a.f.fs) - ld_sub_start(k, a.f.fs) - a.f.lo];
            const double ek[4] = {e[i][0].x, e[i][0].y, e[i][1].x, e[i][1].y};
            double r[4];
#pragma unroll
            for (int row = 0; row < 4; row++)
                r[row] = fma(P[4 * row], s[0], fma(P[4 * row + 1], s[1], fma(P[4 * row + 2], s[2], fma(P[4 * row + 3], s[3], ek[row]))));
#pragma unroll
            for (int row = 0; row < 4; row++) s[row] = r[row];
        }
    }
}

// Tiles of the true-peak pass of an utterance of cnt samples: positions q = -6 .. cnt + 5 in tiles of LD_TP_TILE.
__host__ __device__ __forceinline__ unsigned long long ld_tp_tiles(unsigned long long cnt) {
    return (cnt + 2 * LD_TP_HALO + LD_TP_TILE - 1) / LD_TP_TILE;
}

// Utterance u0 + blockIdx.y, positions q = blockIdx.x * LD_TP_TILE - 6 + [0, LD_TP_TILE): for every q the phases
// v[4q + r] = sum over j = q - 5 .. q + 6 (ascending) of x[j] * h[4(q - j) + r + 24], r = 1 .. 3, one fmaf per term
// from 0.0f, and v[4q] = x[q]; the tile's max |v| goes to tp_tile at the utterance's first tile (off[2(n + 1) + u])
// plus blockIdx.x.  Samples outside [0, cnt) read as zeros, so positions past cnt + 5 add nothing.  The staged
// samples are stored at l + l / 8: thread t reads its 19-sample window l = 8t + 1 .. 8t + 19 at stride 9 words,
// conflict-free.  Every |v| is a non-negative float, whose bits order like its value: the maximum is exact.
__global__ void __launch_bounds__(LD_TP_THREADS) ld_true_peak_kernel(LdArgs a) {
    __shared__ float stage[LD_TP_STAGE + LD_TP_STAGE / 8 + 1];
    __shared__ unsigned red[LD_TP_THREADS / 32];
    const uint32_t u = a.u0 + blockIdx.y;
    const long long cnt = a.counts[u];
    const long long t0 = (long long)blockIdx.x * LD_TP_TILE;
    if ((unsigned long long)t0 >= (unsigned long long)cnt + 2 * LD_TP_HALO) return;   // the whole CTA
    const int16_t* x = a.pcm + a.off[u];
    const long long j0 = t0 - 2 * LD_TP_HALO;   // sample of stage position 0 (positions start at t0 - 6)
    for (uint32_t l = threadIdx.x; l < LD_TP_STAGE; l += LD_TP_THREADS) {
        const long long j = j0 + l;
        stage[l + l / 8] = (j >= 0 && j < cnt) ? (float)x[j] : 0.0f;
    }
    __syncthreads();
    const uint32_t b = LD_TP_PER * threadIdx.x + 1;
    float w[LD_TP_PER + 11];
#pragma unroll
    for (int k = 0; k < LD_TP_PER + 11; k++) w[k] = stage[b + k + (b + k) / 8];
    float m = 0.0f;
#pragma unroll
    for (int p = 0; p < LD_TP_PER; p++) {
        m = fmaxf(m, fabsf(w[p + 5]));   // phase 0: x[q]
#pragma unroll
        for (int r = 0; r < 3; r++) {
            float v = 0.0f;
#pragma unroll
            for (int i = 0; i < 12; i++) v = __fmaf_rn(w[p + i], a.tp_h[r][i], v);
            m = fmaxf(m, fabsf(v));
        }
    }
    const unsigned wm = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
    if ((threadIdx.x & 31u) == 0) red[threadIdx.x >> 5] = wm;
    __syncthreads();
    if (threadIdx.x) return;
    unsigned bits = red[0];
#pragma unroll
    for (int k = 1; k < LD_TP_THREADS / 32; k++) bits = max(bits, red[k]);
    a.tp_tile[a.off[2 * (a.n + 1) + u] + blockIdx.x] = __uint_as_float(bits);
}

// One CTA per utterance: the gated mean of the 400 ms block energies, L, and G = min(table[k], A * 65536 / P) with
// the sample peak P; TRUE_PEAK: G = min(table[k], floor((A - 1) * 65536 / P)) with the true peak P, which is stored.
template <bool TRUE_PEAK>
__global__ void __launch_bounds__(LD_GAIN_THREADS) ld_gain_kernel(LdArgs a) {
    __shared__ double red_d[LD_GAIN_THREADS / 32];
    __shared__ unsigned red_u[LD_GAIN_THREADS / 32];
    const uint32_t u = blockIdx.x;
    const uint32_t cnt = a.counts[u];
    const unsigned long long nch = ld_chunks(a, u, cnt);
    const unsigned long long c0 = a.off[a.n + 1 + u];
    const uint32_t fs = a.f.fs;
    // complete sub-blocks: floor((k + 1) * fs / 10) <= cnt; blocks j = sub-blocks j .. j + 3
    const unsigned long long full = min(((unsigned long long)cnt * 10u + 10u + fs - 1u) / fs - 1u, nch);
    const unsigned long long nb = full >= 4 ? full - 3 : 0;
    unsigned pk = 0;
    if (TRUE_PEAK) {
        const unsigned long long t0 = a.off[2 * (a.n + 1) + u], nt = ld_tp_tiles(cnt);
        for (unsigned long long t = threadIdx.x; t < nt; t += LD_GAIN_THREADS) pk = max(pk, __float_as_uint(a.tp_tile[t0 + t]));
    } else {
        for (unsigned long long k = threadIdx.x; k < nch; k += LD_GAIN_THREADS) pk = max(pk, a.peak[c0 + k]);
    }
    pk = block_allreduce<LD_GAIN_THREADS>(pk, LdMaxU{}, red_u);
    const double* E = a.energy + c0;
    auto z_of = [&](unsigned long long j) {
        return (E[j] + E[j + 1] + E[j + 2] + E[j + 3]) / (double)(ld_sub_start(j + 4, fs) - ld_sub_start(j, fs));
    };
    double sum = 0.0;
    unsigned m = 0;
    for (unsigned long long j = threadIdx.x; j < nb; j += LD_GAIN_THREADS) {
        const double z = z_of(j);
        if (z > a.gate_abs) { sum += z; m++; }
    }
    sum = block_allreduce<LD_GAIN_THREADS>(sum, LdSumD{}, red_d);
    m = block_allreduce<LD_GAIN_THREADS>(m, OpAddU32{}, red_u);
    double sum2 = 0.0;
    unsigned m2 = 0;
    if (m) {
        const double gate_rel = sum / (double)m / 10.0;
        for (unsigned long long j = threadIdx.x; j < nb; j += LD_GAIN_THREADS) {
            const double z = z_of(j);
            if (z > a.gate_abs && z > gate_rel) { sum2 += z; m2++; }
        }
        sum2 = block_allreduce<LD_GAIN_THREADS>(sum2, LdSumD{}, red_d);
        m2 = block_allreduce<LD_GAIN_THREADS>(m2, OpAddU32{}, red_u);
    }
    if (threadIdx.x) return;
    double L = -INFINITY;
    uint32_t G = LD_UNITY;
    if (m2) {
        L = -0.691 + 10.0 * log10(sum2 / (double)m2);
        const double k = fmin(fmax(floor(100.0 * ((double)a.target - L) + 0.5), (double)-LD_K_MAX), (double)LD_K_MAX);
        G = a.table[(int)k + LD_K_MAX];
        if (TRUE_PEAK) {
            // exact operands: (A - 1) * 65536 < 2^31 and a float P; the quotient is rounded once, then floored
            if (pk) G = (uint32_t)fmin((double)G, floor((double)(a.ceiling - 1u) * (double)LD_UNITY / (double)__uint_as_float(pk)));
        } else {
            if (pk) G = (uint32_t)min((unsigned long long)G, (unsigned long long)a.ceiling * LD_UNITY / pk);
        }
    }
    a.lufs[u] = L;
    a.gain[u] = G;
    if (TRUE_PEAK) a.tp_peak[u] = __uint_as_float(pk);
}

// Utterance u0 + blockIdx.y, tile blockIdx.x of LD_APPLY_TILE samples, 16-byte vectors (slots start 16-byte aligned).
// Samples past the count are left as they are.  |y| <= A follows from G <= A * 65536 / P (sample peak) and from the
// true-peak guarantee of DESIGN.md 5: no saturation.
__global__ void __launch_bounds__(LD_APPLY_THREADS) ld_apply_kernel(LdArgs a) {
    const uint32_t u = a.u0 + blockIdx.y;
    const uint32_t G = a.gain[u];
    if (G == LD_UNITY) return;
    const uint32_t cnt = a.counts[u];
    const uint32_t t0 = blockIdx.x * LD_APPLY_TILE;
    if (t0 >= cnt) return;
    int4* p = reinterpret_cast<int4*>(a.pcm + a.off[u]);
    const uint32_t v1 = min((cnt + 7u) >> 3, (t0 + LD_APPLY_TILE) >> 3);
    for (uint32_t v = (t0 >> 3) + threadIdx.x; v < v1; v += LD_APPLY_THREADS) {
        int4 q = __ldcs(p + v);
        int16_t* e = reinterpret_cast<int16_t*>(&q);
#pragma unroll
        for (int k = 0; k < 8; k++)
            if (8u * v + (uint32_t)k < cnt) e[k] = (int16_t)(((long long)e[k] * G + 32768) >> 16);
        __stcs(p + v, q);
    }
}

}  // namespace ctts
