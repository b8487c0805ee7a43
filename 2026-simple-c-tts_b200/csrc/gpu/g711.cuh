// g711.cuh -- G.711 output of the packed session path (DESIGN.md 3.7): every output-rate int16 sample becomes one
// μ-law or A-law byte (ITU-T G.711 as the G.191 tools and Sun's g711.c encode it), in the PCM session's packed
// layout with bytes in place of samples.  pack_scan_kernel's offsets (counts rounded up to 8) are byte offsets here.
//
//   g711_pack_kernel   takes the place of pack_copy_kernel: utterance blockIdx.y, tile blockIdx.x of PACK_TILE
//                      samples; each thread reads 8 samples (16 bytes, streaming), encodes them branch-free and
//                      stores 8 bytes (streaming); the <= 7 bytes of padding get the law's code for silence
#pragma once
#include <cstdint>

#include "assemble.cuh"

namespace ctts {

constexpr int G711_ULAW = 1;   // == CTTS_GPU_G711_ULAW
constexpr int G711_ALAW = 2;   // == CTTS_GPU_G711_ALAW

// The code of 0: what a player hears as silence (a zero byte is near full scale in both laws)
template <int LAW>
__host__ __device__ constexpr uint32_t g711_silence() { return LAW == G711_ULAW ? 0xFFu : 0xD5u; }

// One sample -> one code.  The segment is the position of the magnitude's top bit, from __clz, not a table search.
template <int LAW>
__device__ __forceinline__ uint32_t g711_encode(int x) {
    if (LAW == G711_ULAW) {
        // top 14 bits; magnitude clipped to 8159, bias 33 -> [33, 8192]; segment s: m < 64 << s; 8192 -> 0x7F
        const int v = x >> 2;
        const uint32_t m = (uint32_t)min(abs(v), 8159) + 33u;
        const uint32_t seg = 26u - (uint32_t)__clz((int)m);   // 0 .. 8
        const uint32_t code = min((seg << 4) | ((m >> (seg + 1u)) & 0xFu), 0x7Fu);
        return code ^ (v < 0 ? 0x7Fu : 0xFFu);
    } else {
        // top 13 bits; -v - 1 for negative input -> [0, 4095]; segment s: m < 32 << s; mantissa shift max(s, 1)
        const int v = x >> 3;
        const uint32_t m = (uint32_t)(v < 0 ? ~v : v);
        const uint32_t seg = (uint32_t)max(27 - __clz((int)(m | 1u)), 0);   // 0 .. 7
        const uint32_t code = (seg << 4) | ((m >> max(seg, 1u)) & 0xFu);
        return code ^ (v < 0 ? 0x55u : 0xD5u);
    }
}

// Two samples packed in a 32-bit word (little end first) -> their two codes in the low 16 bits; codes of samples at
// or past `cnt` (k counts from the word's first sample) are the silence code.
template <int LAW>
__device__ __forceinline__ uint32_t g711_pair(uint32_t w, uint32_t k, uint32_t cnt) {
    const uint32_t a = k < cnt ? g711_encode<LAW>((int)(int16_t)(w & 0xFFFFu)) : g711_silence<LAW>();
    const uint32_t b = k + 1u < cnt ? g711_encode<LAW>((int)(int16_t)(w >> 16)) : g711_silence<LAW>();
    return a | (b << 8);
}

template <int LAW>
__global__ void __launch_bounds__(PACK_THREADS) g711_pack_kernel(const int16_t* __restrict__ slots, const unsigned long long* __restrict__ slot_off,
                                                                 const uint32_t* __restrict__ counts, const unsigned long long* __restrict__ pack_off,
                                                                 uint8_t* __restrict__ packed) {
    const uint32_t u = blockIdx.y;
    const uint32_t cnt = counts[u];
    const uint32_t t0 = blockIdx.x * PACK_TILE;
    if (t0 >= cnt) return;
    const int4* src = reinterpret_cast<const int4*>(slots + slot_off[u]);
    uint2* dst = reinterpret_cast<uint2*>(packed + pack_off[u]);
    const uint32_t nvec = (cnt + 7u) >> 3;
    const uint32_t v1 = min(nvec, (t0 + PACK_TILE) >> 3);
    for (uint32_t v = (t0 >> 3) + threadIdx.x; v < v1; v += PACK_THREADS) {
        const int4 q = __ldcs(src + v);
        const uint32_t k = 8u * v;
        const uint32_t lo = g711_pair<LAW>((uint32_t)q.x, k, cnt) | (g711_pair<LAW>((uint32_t)q.y, k + 2u, cnt) << 16);
        const uint32_t hi = g711_pair<LAW>((uint32_t)q.z, k + 4u, cnt) | (g711_pair<LAW>((uint32_t)q.w, k + 6u, cnt) << 16);
        __stcs(dst + v, make_uint2(lo, hi));
    }
}

}  // namespace ctts
