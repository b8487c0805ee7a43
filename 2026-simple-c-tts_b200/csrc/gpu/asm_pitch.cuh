// asm_pitch.cuh -- pitch smoothing at joins (ctts.c:1899-2024).
#pragma once
#include "asm_common.cuh"

namespace ctts {

// ---------------------------------------------------------------- pitch

// estimate_pitch (ctts.c:1899) for two signals of the same length at once (the
// buffer tail `a` and the unit head `b`).
//
// The reference evaluates, for each lag in 55..275, three sequential float sums
// over i < 220: corr += s[i]*s[i+lag], e1 += s[i]^2, e2 += s[i+lag]^2, and keeps
// the first lag whose corr/sqrtf(e1*e2) is the strict maximum (voiced iff > 0.3).
// Those sums cannot be reordered, and at 3 non-fused FP32 operations per
// (lag, i) pair they would be 40 % of all instructions of the assembly path.  So
// the search is done in two steps that together give the identical result:
//
//  1. FILTER: every lag gets an approximate score a[lag] = c~ / sqrtf(e1x * e2x),
//     c~ accumulated with FMA (one instruction per pair, four lags per thread
//     sharing the operand loads, the i range split over two threads) and e1x, e2x
//     EXACT integer window sums taken from a 64-bit prefix sum of the squares.
//     For 220 terms |a - r| <= 4.0e-5 where r is the reference's score (standard
//     summation error bound, gamma_n * sum|x_i*y_i| <= gamma_n * sqrt(e1*e2) by
//     Cauchy-Schwarz; DESIGN.md derives it).
//  2. DECIDE: with eps = 1e-4 (3 x the rigorous worst-case bound 3.4e-5) a signal is unvoiced if
//     max a <= 0.3 - eps.  Otherwise only lags with a >= max a - 2*eps can be the
//     reference's arg max.  If that is a single lag and its score exceeds
//     0.3 + eps, the answer is known.  Else the candidates (typically 2-3) are
//     evaluated by one thread each with the reference's exact operation order.
//
// Both signals are needed voiced by the caller, so step 2 is skipped entirely
// when either signal fails the filter.
//
// pair == false: only signal `a` is estimated (the threads of signal b idle).  The pitch of an
// untouched unit head over a given analysis length is a function of the voice alone and comes
// from a table (unit_pitch_kernel below), which leaves the buffer tail as the only signal.
constexpr int PITCH_LO = CTTS_PLAN_SAMPLE_RATE / 400;  // 55
constexpr int PITCH_HI = CTTS_PLAN_SAMPLE_RATE / 80;   // 275
constexpr int PITCH_LEN = CTTS_PLAN_SAMPLE_RATE / 100; // 220
constexpr int PITCH_LAG0 = 53;        // lag of thread 0 (= 1 mod 4 keeps both float4 loads aligned)
constexpr int PITCH_LPT = 4;          // lags per thread
constexpr int PITCH_TPS = 64;         // threads per signal and half (57 used)
constexpr int PITCH_Y = 512;          // staged floats per signal (zero padded)
constexpr int PITCH_S = 512;          // prefix entries per signal
constexpr int PITCH_MAX_CAND = 64;    // per signal, beyond that: every lag is evaluated exactly
constexpr float PITCH_EPS = 1e-4f;
constexpr int PITCH_SCRATCH_WORDS = 2 * PITCH_Y + 2 * 2 * PITCH_S + 4 + 2 * (PITCH_MAX_CAND + 2) + 16 + 4 * 2 * PITCH_TPS;
static_assert(ASM_THREADS == 4 * PITCH_TPS, "2 signals x 2 halves x PITCH_TPS threads");
static_assert(PITCH_LAG0 % 4 == 1 && PITCH_LAG0 <= PITCH_LO, "lag tiling");
static_assert(PITCH_SCRATCH_WORDS <= (int)SCR_WORDS, "pitch scratch fits");
static_assert(PITCH_LAG0 + PITCH_LPT * 57 > PITCH_HI, "57 threads cover every lag");
static_assert(PITCH_HI + PITCH_LPT + PITCH_LEN + 8 <= PITCH_Y, "staging covers the loop's reads");
static_assert(PITCH_HI + PITCH_LEN < PITCH_S, "prefix covers every window");

// exact sums of one lag in the reference's order (ctts.c:1917-1931); lag 0 yields e1 in *e2_out
__device__ __forceinline__ float pitch_exact_sums(const float* y, uint32_t lag, uint32_t len, float* e2_out) {
    float c = 0.0f, e2 = 0.0f;
    const float* x = y;
    const float* z = y + lag;
#pragma unroll 4
    for (uint32_t i = 0; i < len; i++) {
        const float a = x[i], b = z[i];
        c += a * b;
        e2 += b * b;
    }
    *e2_out = e2;
    return c;
}

// S[i] = sum_{j<i} s[j]^2 for i < PITCH_S, exact (int16 inputs, 512 * 2^30 < 2^64); one warp.
// A lane owns four groups of four consecutive samples, group q at 4 * (lane + 32 q): consecutive
// lanes touch consecutive 8-byte (input) / 32-byte (output) pieces, so neither the loads nor the
// 16-byte stores collide on a bank (a contiguous 16-sample run per lane would collide 8-16 way).
__device__ __forceinline__ void pitch_prefix_warp(const int16_t* s, uint32_t need, unsigned long long* S) {
    const int lane = lane_id();
    int v[4][4];
    unsigned long long rs[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const uint32_t i0 = 4u * (uint32_t)(lane + 32 * q);
        rs[q] = 0;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            v[q][c] = i0 + c < need ? (int)s[i0 + c] : 0;
            rs[q] += (unsigned long long)(uint32_t)(v[q][c] * v[q][c]);
        }
    }
    unsigned long long carry = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        unsigned long long inc = rs[q];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        unsigned long long run = carry + inc - rs[q];   // exclusive prefix at the lane's first sample
        carry += __shfl_sync(0xffffffffu, inc, 31);
        ulonglong2 lo, hi;
        lo.x = run; run += (unsigned long long)(uint32_t)(v[q][0] * v[q][0]);
        lo.y = run; run += (unsigned long long)(uint32_t)(v[q][1] * v[q][1]);
        hi.x = run; run += (unsigned long long)(uint32_t)(v[q][2] * v[q][2]);
        hi.y = run;
        ulonglong2* dst = reinterpret_cast<ulonglong2*>(S + 4 * (lane + 32 * q));
        dst[0] = lo;
        dst[1] = hi;
    }
}

__device__ void estimate_pitch_pair(const Smem& sm, const int16_t* a, const int16_t* b, uint32_t n,
                                    float* pa, float* pb, const bool pair = true) {
    *pa = 0.0f;
    *pb = 0.0f;
    if (n < 200) return;
    const int tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const uint32_t lo = PITCH_LO;
    uint32_t hi = PITCH_HI;
    if (hi > n / 2) hi = n / 2;
    uint32_t len = PITCH_LEN;
    if (len > n - hi) len = n - hi;
    const uint32_t need = len + hi;  // <= 495 samples of each signal are ever read

    float* ya = reinterpret_cast<float*>(sm.scratch);
    float* yb = ya + PITCH_Y;
    unsigned long long* Sa = reinterpret_cast<unsigned long long*>(yb + PITCH_Y);  // 8-byte aligned: 2*PITCH_Y even
    unsigned long long* Sb = Sa + PITCH_S;
    unsigned long long* keys = Sb + PITCH_S;                      // [2]
    uint32_t* cand = reinterpret_cast<uint32_t*>(keys + 2);       // [2][PITCH_MAX_CAND + 2]
    uint32_t* ncand = cand + 2 * (PITCH_MAX_CAND + 2);            // [2]
    float* amax = reinterpret_cast<float*>(ncand + 2);            // [4] per lag warp
    float* e1s = amax + 4;                                        // [2]
    float4* cpart = reinterpret_cast<float4*>(e1s + 10);          // [2 * PITCH_TPS] partial sums of the second halves

    // ---- warps 0-1: exact prefix sums of squares; warps 2-7: float staging
    if (warp == 0) pitch_prefix_warp(a, need, Sa);
    else if (warp == 1) {
        if (pair) pitch_prefix_warp(b, need, Sb);
    } else {
        for (uint32_t i = tid - 64; i < (pair ? 2u : 1u) * PITCH_Y; i += ASM_THREADS - 64) {
            const uint32_t k = i & (PITCH_Y - 1);
            const int16_t* src = i < PITCH_Y ? a : b;
            ya[i] = k < need ? (float)src[k] : 0.0f;   // yb == ya + PITCH_Y
        }
        if (tid < 66) {
            ncand[tid - 64] = 0;
            keys[tid - 64] = 0ull;
        }
    }
    __syncthreads();

    // ---- step 1: FMA scores; thread (part, signal, lag group) accumulates its part of the i range:
    //      two signals x two halves, or one signal x four quarters
    float c[PITCH_LPT] = {0.0f, 0.0f, 0.0f, 0.0f};
    const int part = pair ? tid >> 7 : tid >> 6;
    const int sig = pair ? (tid >> 6) & 1 : 0;
    const uint32_t lag0 = PITCH_LAG0 + PITCH_LPT * (uint32_t)(tid & (PITCH_TPS - 1));
    const bool lag_thread = lag0 <= hi;
    // part boundaries are multiples of 4: every part keeps the float4 alignment; the parts cover all len terms
    const uint32_t step = pair ? (((len + 1u) >> 1) + 3u) & ~3u : (((len + 3u) >> 2) + 3u) & ~3u;
    if (!pair) cpart = reinterpret_cast<float4*>(Sb);   // signal b's prefix array is free: 3 x PITCH_TPS partials
    if (lag_thread) {
        const float* x = sig ? yb : ya;
        const float* y = x + lag0;  // y[j] = s[lag0 + j]; (lag0 + 3) % 4 == 0
        const uint32_t i_begin = min((uint32_t)part * step, len);
        const uint32_t i_end = min(i_begin + step, len);
        if (i_begin < i_end) {
            float w0 = y[i_begin], w1 = y[i_begin + 1], w2 = y[i_begin + 2];
            const uint32_t i4 = i_begin + ((i_end - i_begin) & ~3u);
            for (uint32_t i = i_begin; i < i4; i += 4) {
                const float4 xv = *reinterpret_cast<const float4*>(x + i);
                const float4 yn = *reinterpret_cast<const float4*>(y + i + 3);
                const float w3 = yn.x, w4 = yn.y, w5 = yn.z, w6 = yn.w;
                c[0] = __fmaf_rn(xv.x, w0, c[0]); c[1] = __fmaf_rn(xv.x, w1, c[1]);
                c[2] = __fmaf_rn(xv.x, w2, c[2]); c[3] = __fmaf_rn(xv.x, w3, c[3]);
                c[0] = __fmaf_rn(xv.y, w1, c[0]); c[1] = __fmaf_rn(xv.y, w2, c[1]);
                c[2] = __fmaf_rn(xv.y, w3, c[2]); c[3] = __fmaf_rn(xv.y, w4, c[3]);
                c[0] = __fmaf_rn(xv.z, w2, c[0]); c[1] = __fmaf_rn(xv.z, w3, c[1]);
                c[2] = __fmaf_rn(xv.z, w4, c[2]); c[3] = __fmaf_rn(xv.z, w5, c[3]);
                c[0] = __fmaf_rn(xv.w, w3, c[0]); c[1] = __fmaf_rn(xv.w, w4, c[1]);
                c[2] = __fmaf_rn(xv.w, w5, c[2]); c[3] = __fmaf_rn(xv.w, w6, c[3]);
                w0 = w4; w1 = w5; w2 = w6;
            }
            for (uint32_t i = i4; i < i_end; i++) {
                const float xs = x[i];
#pragma unroll
                for (int k = 0; k < PITCH_LPT; k++) c[k] = __fmaf_rn(xs, y[i + k], c[k]);
            }
        }
        if (part) cpart[pair ? (tid & (2 * PITCH_TPS - 1)) : (part - 1) * PITCH_TPS + (tid & (PITCH_TPS - 1))] = make_float4(c[0], c[1], c[2], c[3]);
    }
    __syncthreads();

    // ---- scores and per-signal maximum (part 0 threads)
    float sc[PITCH_LPT];
    float my_max = -1.0f;
    if (lag_thread && !part) {
        for (int q = 0; q < (pair ? 1 : 3); q++) {
            const float4 p2 = cpart[q * PITCH_TPS + tid];   // pair: tid < 128, one partial
            c[0] += p2.x; c[1] += p2.y; c[2] += p2.z; c[3] += p2.w;
        }
        const unsigned long long* S = sig ? Sb : Sa;
        const float e1 = (float)(S[len] - S[0]);
#pragma unroll
        for (int k = 0; k < PITCH_LPT; k++) {
            const uint32_t lag = lag0 + k;
            sc[k] = -1.0f;
            if (lag >= lo && lag <= hi) {
                const float e2 = (float)(S[lag + len] - S[lag]);
                const float nn = e1 * e2;   // exact integers >= 1 when nonzero; the filter may use rsqrt.approx (2^-22)
                sc[k] = nn > 0.0f ? c[k] * rsqrt_approx(nn) : 0.0f;
                my_max = fmaxf(my_max, sc[k]);
            }
        }
    }
    if (tid < 2 * PITCH_TPS) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_max = fmaxf(my_max, __shfl_xor_sync(0xffffffffu, my_max, o));
        if (lane == 0) amax[warp] = my_max;
    }
    __syncthreads();
    const float max_a = fmaxf(amax[0], amax[1]), max_b = pair ? fmaxf(amax[2], amax[3]) : 1.0f;
    // unvoiced by the filter: the reference's best cannot exceed 0.3
    if (!(max_a > 0.3f - PITCH_EPS) || !(max_b > 0.3f - PITCH_EPS)) {   // CTA-uniform
        __syncthreads();   // scratch is reused by the caller
        return;
    }

    // ---- candidates
    if (lag_thread && !part) {
        const float thr = (sig ? max_b : max_a) - 2.0f * PITCH_EPS;
#pragma unroll
        for (int k = 0; k < PITCH_LPT; k++) {
            if (sc[k] >= thr) {
                uint32_t slot = atomicAdd(ncand + sig, 1u);
                if (slot < PITCH_MAX_CAND) cand[sig * (PITCH_MAX_CAND + 2) + slot] = lag0 + k;
            }
        }
    }
    __syncthreads();
    uint32_t na = ncand[0], nb = ncand[1];
    // a single candidate well above the voicing threshold IS the reference's answer
    const bool sure_a = na == 1 && max_a > 0.3f + PITCH_EPS, sure_b = !pair || (nb == 1 && max_b > 0.3f + PITCH_EPS);
    if (sure_a) *pa = (float)CTTS_PLAN_SAMPLE_RATE / (float)cand[0];
    if (sure_b && pair) *pb = (float)CTTS_PLAN_SAMPLE_RATE / (float)cand[PITCH_MAX_CAND + 2];
    if (sure_a && sure_b) {
        __syncthreads();
        return;
    }
    const bool all_a = na > PITCH_MAX_CAND, all_b = nb > PITCH_MAX_CAND;  // degenerate: evaluate every lag
    if (all_a) na = hi - lo + 1;
    if (all_b) nb = hi - lo + 1;
    if (sure_a) na = 0;   // nothing to evaluate for a settled signal
    if (sure_b) nb = 0;
    __syncthreads();

    // ---- step 2: exact evaluation, one thread per (signal, lag); job 0 of each signal is lag 0 (= e1)
    const uint32_t ja = sure_a ? 0u : na + 1, jb = sure_b ? 0u : nb + 1;
    const uint32_t jobs = ja + jb;
    for (uint32_t j = tid; j < jobs; j += ASM_THREADS) {
        const int sg = j < ja ? 0 : 1;
        const uint32_t jj = sg ? j - ja : j;
        if (jj == 0) {
            float e1;
            (void)pitch_exact_sums(sg ? yb : ya, 0, len, &e1);
            e1s[sg] = e1;
        } else {
            const bool all = sg ? all_b : all_a;
            const uint32_t lag = all ? lo + (jj - 1) : cand[sg * (PITCH_MAX_CAND + 2) + (jj - 1)];
            float e2;
            const float cc = pitch_exact_sums(sg ? yb : ya, lag, len, &e2);
            // park the raw sums; the score needs e1, which another thread is computing
            reinterpret_cast<float2*>(sg ? Sb : Sa)[jj] = make_float2(cc, e2);   // S is dead from here on
        }
    }
    __syncthreads();
    for (uint32_t j = tid; j < jobs; j += ASM_THREADS) {
        const int sg = j < ja ? 0 : 1;
        const uint32_t jj = sg ? j - ja : j;
        if (jj == 0) continue;
        const bool all = sg ? all_b : all_a;
        const uint32_t lag = all ? lo + (jj - 1) : cand[sg * (PITCH_MAX_CAND + 2) + (jj - 1)];
        const float2 ce = reinterpret_cast<const float2*>(sg ? Sb : Sa)[jj];
        float v = ce.x;
        const float nrm = sqrtf(e1s[sg] * ce.y);
        if (nrm > 0) v /= nrm;
        // the reference keeps the first lag that is strictly greater than everything before it,
        // starting from 0: the maximum positive score, smallest lag on ties
        if (v > 0.0f) atomicMax(keys + sg, ((unsigned long long)__float_as_uint(v) << 32) | (0xffffffffu - lag));
    }
    __syncthreads();
    const unsigned long long ka = keys[0], kb = keys[1];
    if (!sure_a) {
        const float v = __uint_as_float((uint32_t)(ka >> 32));
        const uint32_t l = 0xffffffffu - (uint32_t)(ka & 0xffffffffu);
        if (ka != 0ull && v > 0.3f && l > 0) *pa = (float)CTTS_PLAN_SAMPLE_RATE / (float)l;
    }
    if (!sure_b) {
        const float v = __uint_as_float((uint32_t)(kb >> 32));
        const uint32_t l = 0xffffffffu - (uint32_t)(kb & 0xffffffffu);
        if (kb != 0ull && v > 0.3f && l > 0) *pb = (float)CTTS_PLAN_SAMPLE_RATE / (float)l;
    }
    __syncthreads();   // scratch is reused by the caller
}

// estimate_pitch (ctts.c:1899) of the first job.y samples of the normalized unit at pool offset
// job.x, into table[job.z]: what smooth_pitch_boundary computes for `next_samples` whenever the
// analysis length is min(2*xf, n/2).  One CTA per (unit, length) pair the plan compiler has not
// seen in this context before.
__global__ void __launch_bounds__(ASM_THREADS) unit_pitch_kernel(const int16_t* __restrict__ norm_pool, const uint3* __restrict__ jobs,
                                                                 float* __restrict__ table) {
    __shared__ __align__(16) uint32_t scratch[SCR_WORDS];
    Smem sm{};
    sm.scratch = scratch;
    const uint3 job = jobs[blockIdx.x];
    const int16_t* head = norm_pool + job.x;
    float pa = 0.0f, pb = 0.0f;
    estimate_pitch_pair(sm, head, head, job.y, &pa, &pb, false);
    if (threadIdx.x == 0) table[job.z] = pa;
}

// smooth_pitch_boundary + apply_pitch_shift, ctts.c:1946-2024.  `reg` is the analysis length
// min(2*xf, count/2, n/2) resolved by the caller (0 = the reference returns early); `us` is the
// staged unit head; have_np: the head's pitch over `reg` samples is the table value np_tab.
__device__ void smooth_pitch(const State& s, const Smem& sm, int16_t* us, uint32_t n, uint32_t xf, uint32_t reg,
                             bool have_np, float np_tab) {
    if (reg == 0) return;
    const int tid = threadIdx.x;
    float pp, np;
    const int16_t* prev = s.w + ((int)s.cnt - (int)reg);
    if (have_np) {
        np = np_tab;
        if (!(np > 0)) return;   // ctts.c:1994: both must be voiced
        float unused;
        estimate_pitch_pair(sm, prev, prev, reg, &pp, &unused, false);
    } else {
        estimate_pitch_pair(sm, prev, us, reg, &pp, &np);
    }
    if (!(pp > 0 && np > 0)) return;
    float ratio = np / pp;
    if (!(ratio > 1.15f || ratio < 0.85f)) return;
    float target = (ratio > 1.0f) ? 1.0f + (ratio - 1.0f) * 0.5f : 1.0f - (1.0f - ratio) * 0.5f;
    float shift = target / ratio;
    uint32_t len = xf;
    if (len > n / 4) len = n / 4;
    int16_t* tmp = reinterpret_cast<int16_t*>(sm.scratch);  // len <= hcap <= 2 * SCR_WORDS (host check)
    bool do_shift = !(shift < 0.9f || shift > 1.1f || len < 100);
    uint32_t keep = len;
    if (do_shift) {
        uint32_t m = (uint32_t)(unsigned long long)((float)len / shift);
        keep = m < len ? m : len;
    }
    for (uint32_t i = tid; i < len; i += ASM_THREADS) {
        int16_t r = 0;
        if (!do_shift) {
            r = us[i];
        } else if (i < keep) {
            float x = (float)i * shift;
            uint32_t k = (uint32_t)(unsigned long long)x;
            float fr = x - (float)k;
            if (k + 1 < len) r = f2s((float)us[k] * (1.0f - fr) + (float)us[k + 1] * fr);
            else if (k < len) r = us[k];
        }
        tmp[i] = r;
    }
    __syncthreads();
    const float flen = (float)len, rlen = recip_for_div(flen);
    for (uint32_t i = tid; i < len; i += ASM_THREADS) {
        const float t = div_by((float)i, flen, rlen);
        us[i] = f2s((float)tmp[i] * (1.0f - t) + (float)us[i] * t);
    }
    __syncthreads();
}

// match_boundary_energy, ctts.c:1730 (sums of squares are exact integers); len = min(xf, count, n)
__device__ void match_energy(const State& s, const Smem& sm, int16_t* us, uint32_t len) {
    if (len == 0) return;
    const int tid = threadIdx.x;
    const int16_t* tail = s.w + ((int)s.cnt - (int)len);
    long long sp = sumsq_range(tail, len), sn = sumsq_range(us, len);
    // ratio = clamp(prev_rms / next_rms) with both rms values in double (ctts.c:1741-1749): one thread
    const unsigned long long rr = block_sum2_then<ASM_THREADS>(sp, sn, reinterpret_cast<long long*>(sm.red), [&](long long tp, long long tn) {
        const float pr = (float)sqrt((double)tp / (double)len);
        const float nr = (float)sqrt((double)tn / (double)len);
        if (pr < 1.0f || nr < 1.0f) return 0ull;
        float ratio = pr / nr;
        if (ratio > 2.0f) ratio = 2.0f;
        if (ratio < 0.5f) ratio = 0.5f;
        return (1ull << 32) | (unsigned long long)__float_as_uint(ratio);
    });
    if ((rr >> 32) == 0) return;
    const float ratio = __uint_as_float((uint32_t)rr);
    // two samples per step (us is 4-byte aligned); t = i / len with the hoisted reciprocal
    const float flen = (float)len, rlen = recip_for_div(flen);
    uint32_t* us2 = reinterpret_cast<uint32_t*>(us);
    for (uint32_t h = tid; 2 * h < len; h += ASM_THREADS) {
        const uint32_t i = 2 * h;
        const uint32_t w = us2[h];
        const float t0 = div_by((float)i, flen, rlen);
        const float g0 = ratio * (1.0f - t0) + 1.0f * t0;
        const int y0 = cvt_sat_s16((float)(short)(w & 0xffffu) * g0);
        int y1 = (int)(short)(w >> 16);
        if (i + 1 < len) {
            const float t1 = div_by((float)(i + 1), flen, rlen);
            const float g1 = ratio * (1.0f - t1) + 1.0f * t1;
            y1 = cvt_sat_s16((float)y1 * g1);
        }
        us2[h] = (uint32_t)(y0 & 0xffff) | ((uint32_t)y1 << 16);
    }
    __syncthreads();
}


}  // namespace ctts
