// block_prims.cuh -- CTA-wide reductions and scans built on warp shuffles.
//
// The assembly path needs exact integer reductions (sums of squares and DC sums
// are order-free because they are integers: SURVEY.md 7.3) and max/min scans for
// the silence-run analysis; float sums are NEVER reduced in parallel anywhere in
// this back end because the reference's float accumulations are sequential.  (The loudness measurement of
// loudness.cuh is the one exception: it is not part of the reference, and its contract carries a tolerance.)
#pragma once
#include <cstdint>

namespace ctts {

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

struct OpAddU64 {
    __device__ __forceinline__ unsigned long long operator()(unsigned long long a, unsigned long long b) const {
        return a + b;
    }
};
struct OpAddI64 {
    __device__ __forceinline__ long long operator()(long long a, long long b) const { return a + b; }
};
struct OpMaxI32 {
    __device__ __forceinline__ int operator()(int a, int b) const { return a > b ? a : b; }
};
struct OpMinI32 {
    __device__ __forceinline__ int operator()(int a, int b) const { return a < b ? a : b; }
};
struct OpAddU32 {
    __device__ __forceinline__ unsigned operator()(unsigned a, unsigned b) const { return a + b; }
};
struct OpMaxU64 {
    __device__ __forceinline__ unsigned long long operator()(unsigned long long a, unsigned long long b) const {
        return a > b ? a : b;
    }
};

// All-reduce over the CTA.  `red` is shared scratch with >= NT/32 entries of V.
// Two barriers; every thread returns the same value.
template <int NT, typename V, typename Op>
__device__ __forceinline__ V block_allreduce(V v, Op op, V* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (lane_id() == 0) red[warp_id()] = v;
    __syncthreads();
    V r = red[0];
#pragma unroll
    for (int k = 1; k < NT / 32; k++) r = op(r, red[k]);
    __syncthreads();
    return r;
}

// Sum of two 64-bit integers per thread in one pass (one barrier pair instead of two).
// `red` needs 2 * NT/32 entries.
template <int NT>
__device__ __forceinline__ void block_allreduce_add2(long long& a, long long& b, long long* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane_id() == 0) {
        red[warp_id()] = a;
        red[NT / 32 + warp_id()] = b;
    }
    __syncthreads();
    long long ra = 0, rb = 0;
#pragma unroll
    for (int k = 0; k < NT / 32; k++) {
        ra += red[k];
        rb += red[NT / 32 + k];
    }
    __syncthreads();
    a = ra;
    b = rb;
}

// Sum of one (or two) 64-bit integers per thread; THREAD 0 ALONE maps the total(s) through fn --
// the FP64 / 64-bit-division work that follows such a sum would otherwise be repeated by every
// thread -- and the 64-bit result is broadcast.  Two barriers, like block_allreduce.
// `red` needs 2 * NT/32 + 1 entries.
template <int NT, typename F>
__device__ __forceinline__ unsigned long long block_sum_then(long long a, long long* red, F fn) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane_id() == 0) red[warp_id()] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
#pragma unroll
        for (int k = 0; k < NT / 32; k++) t += red[k];
        reinterpret_cast<unsigned long long*>(red)[2 * (NT / 32)] = fn(t);
    }
    __syncthreads();
    return reinterpret_cast<unsigned long long*>(red)[2 * (NT / 32)];
}
template <int NT, typename F>
__device__ __forceinline__ unsigned long long block_sum2_then(long long a, long long b, long long* red, F fn) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane_id() == 0) {
        red[warp_id()] = a;
        red[NT / 32 + warp_id()] = b;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        long long ta = 0, tb = 0;
#pragma unroll
        for (int k = 0; k < NT / 32; k++) {
            ta += red[k];
            tb += red[NT / 32 + k];
        }
        reinterpret_cast<unsigned long long*>(red)[2 * (NT / 32)] = fn(ta, tb);
    }
    __syncthreads();
    return reinterpret_cast<unsigned long long*>(red)[2 * (NT / 32)];
}

// Exclusive scan of one value per thread in thread order (reverse = suffix scan).
// Op must be commutative and associative.  Optionally returns the CTA total.
template <int NT, typename V, typename Op>
__device__ __forceinline__ V block_excl_scan(V v, Op op, V ident, V* red, bool reverse, V* total = nullptr) {
    const int lane = lane_id(), warp = warp_id();
    V x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        V y = reverse ? __shfl_down_sync(0xffffffffu, x, o) : __shfl_up_sync(0xffffffffu, x, o);
        bool ok = reverse ? (lane + o < 32) : (lane >= o);
        if (ok) x = op(x, y);
    }
    if (lane == (reverse ? 0 : 31)) red[warp] = x;
    V ex = reverse ? __shfl_down_sync(0xffffffffu, x, 1) : __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == (reverse ? 31 : 0)) ex = ident;
    __syncthreads();
    V pre = ident;
    V all = ident;
#pragma unroll
    for (int k = 0; k < NT / 32; k++) {
        V r = red[k];
        all = op(all, r);
        bool before = reverse ? (k > warp) : (k < warp);
        if (before) pre = op(pre, r);
    }
    __syncthreads();
    if (total) *total = all;
    return op(pre, ex);
}

}  // namespace ctts
