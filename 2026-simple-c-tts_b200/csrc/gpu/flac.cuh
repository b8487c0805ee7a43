// flac.cuh -- FLAC output of the packed session path (DESIGN.md 3.5): every utterance becomes one self-contained
// .flac file (RFC 9639), mono, 16 bit, fixed blocksize 4096, CONSTANT / VERBATIM / FIXED subframes with Rice
// method 0.  The encoder's choices are exact integer rules, so tests/flac_oracle.c restates them byte for byte.
//
//   flac_analyze_kernel   one CTA per (utterance, frame): subframe kind, fixed order, partition order and Rice
//                         parameters, and the frame's byte length -> a FlacFrame descriptor
//   flac_scan_kernel      one CTA: per utterance the file size (42 + its frames), the frames' offsets inside the
//                         file, min / max frame size; across utterances the packed byte offsets (16-byte aligned);
//                         counts, flags and sizes go straight into page-locked host memory (like pack_scan_kernel)
//   flac_emit_kernel      one CTA per (utterance, frame): assembles the frame's bits in shared memory, CRC-8 of the
//                         header, CRC-16 of the frame, stores it at its byte offset; frame 0's CTA also writes
//                         "fLaC" + STREAMINFO and zeroes the alignment padding behind the file
#pragma once
#include <cstdint>

#include "block_prims.cuh"

namespace ctts {

constexpr uint32_t FLAC_BLOCK = 4096;        // samples per frame (the last frame holds the remainder)
constexpr int FLAC_THREADS = 256;            // 16 samples per thread
constexpr int FLAC_PER_THREAD = FLAC_BLOCK / FLAC_THREADS;
constexpr int FLAC_MAX_PO = 8;               // partition orders 0..8: at most 256 partitions
constexpr int FLAC_KMAX = 14;                // Rice parameters 0..14 (4-bit, 15 is the escape code)
constexpr uint32_t FLAC_HEADER_BYTES = 42;   // "fLaC" + STREAMINFO
constexpr uint32_t FLAC_FRAME_MAX = 16 + 1 + 2 * FLAC_BLOCK + 2;   // header bound + VERBATIM subframe + CRC-16

enum : uint8_t { FLAC_CONSTANT = 0, FLAC_VERBATIM = 1, FLAC_FIXED = 2 };

struct FlacFrame {
    uint32_t bytes;     // frame length in bytes
    uint32_t off;       // byte offset of the frame inside its file (flac_scan_kernel)
    uint8_t kind, order, po, pad;
    uint8_t k[1 << FLAC_MAX_PO];   // Rice parameter of every partition
};

struct FlacArgs {
    const int16_t* slots;                  // output-rate slots
    const unsigned long long* slot_off;    // n + 1
    const uint32_t* counts;
    const unsigned long long* frame_base;  // n + 1: first descriptor of every utterance
    FlacFrame* frames;
    unsigned long long* byte_off;          // n + 1: packed byte offsets (flac_scan_kernel)
    uint32_t* uinfo;                       // 3n: file bytes, min frame bytes, max frame bytes
    uint8_t* out;                          // packed files
    uint32_t hz;                           // sample rate of the STREAMINFO and the frame headers
};

// ---------------------------------------------------------------- shared helpers (host-mirrored in flac_oracle.c)

__device__ __forceinline__ uint32_t flac_rate_code(uint32_t hz) {
    switch (hz) {
        case 8000: return 4;
        case 16000: return 5;
        case 22050: return 6;
        case 24000: return 7;
        case 32000: return 8;
        case 44100: return 9;
        case 48000: return 10;
        default: return 13;   // 16-bit Hz at the end of the header
    }
}

// Frame header without and with its CRC-8: sync 0xFFF8, blocksize code, rate code, mono, 16 bit, the frame number
// in the UTF-8-like coding, the blocksize - 1 of a short frame, the 16-bit rate.  Returns the length (<= 16 bytes).
__device__ __forceinline__ uint32_t flac_frame_header(uint8_t* h, uint32_t frame, uint32_t n, uint32_t hz) {
    const uint32_t rc = flac_rate_code(hz);
    const uint32_t bc = n == FLAC_BLOCK ? 12u : (n - 1 < 256 ? 6u : 7u);
    uint32_t p = 0;
    h[p++] = 0xFF;
    h[p++] = 0xF8;
    h[p++] = (uint8_t)(bc << 4 | rc);
    h[p++] = 0x08;   // channel assignment 0000 (mono), sample size 100 (16 bit), reserved 0
    if (frame < 0x80) {
        h[p++] = (uint8_t)frame;
    } else {
        int extra = frame < 0x800 ? 1 : frame < 0x10000 ? 2 : frame < 0x200000 ? 3 : frame < 0x4000000 ? 4 : 5;
        h[p++] = (uint8_t)((0xFF00u >> (extra + 1)) | (frame >> (6 * extra)));
        for (int i = extra - 1; i >= 0; i--) h[p++] = (uint8_t)(0x80 | ((frame >> (6 * i)) & 0x3F));
    }
    if (bc == 6) h[p++] = (uint8_t)(n - 1);
    if (bc == 7) {
        h[p++] = (uint8_t)((n - 1) >> 8);
        h[p++] = (uint8_t)(n - 1);
    }
    if (rc == 13) {
        h[p++] = (uint8_t)(hz >> 8);
        h[p++] = (uint8_t)hz;
    }
    uint32_t crc = 0;
    for (uint32_t i = 0; i < p; i++) {
        crc ^= h[i];
        for (int b = 0; b < 8; b++) crc = (crc & 0x80) ? ((crc << 1) ^ 0x07) & 0xFF : (crc << 1) & 0xFF;
    }
    h[p++] = (uint8_t)crc;
    return p;
}

__device__ __forceinline__ int flac_residual(const int16_t* x, uint32_t i, uint32_t order) {
    const int a = x[i];
    switch (order) {
        case 0: return a;
        case 1: return a - x[i - 1];
        case 2: return a - 2 * x[i - 1] + x[i - 2];
        case 3: return a - 3 * x[i - 1] + 3 * x[i - 2] - x[i - 3];
        default: return a - 4 * x[i - 1] + 6 * x[i - 2] - 4 * x[i - 3] + x[i - 4];
    }
}
__device__ __forceinline__ uint32_t flac_zigzag(int r) { return r >= 0 ? 2u * (uint32_t)r : 2u * (uint32_t)(-r) - 1u; }

// The utterance's frames that exist: its count, clamped to its slot (a count past the slot comes with a device
// error flag, and the kernels must still stay inside the buffers).
__device__ __forceinline__ uint32_t flac_count(const FlacArgs& a, uint32_t u) {
    return (uint32_t)min((unsigned long long)a.counts[u], a.slot_off[u + 1] - a.slot_off[u]);
}

// ---------------------------------------------------------------- analysis

struct FlacAnalyzeSmem {
    union {
        int16_t x[FLAC_BLOCK];
        uint32_t zz[FLAC_BLOCK];   // zigzag residuals of the chosen order (from index `order` on)
    };
    unsigned long long s[(1 << FLAC_MAX_PO) * (FLAC_KMAX + 1)];   // per partition and k: sum of u >> k
    uint8_t kb[(2 << FLAC_MAX_PO) - 1];                           // best k per partition, all levels (1 << po) - 1 + j
    unsigned long long red[2 * (FLAC_THREADS / 32) + 1];
    unsigned long long level_bits[FLAC_MAX_PO + 1];
};

__global__ void __launch_bounds__(FLAC_THREADS) flac_analyze_kernel(FlacArgs a, uint32_t u_base) {
    __shared__ FlacAnalyzeSmem sm;
    const uint32_t u = u_base + blockIdx.y, f = blockIdx.x, tid = threadIdx.x;
    const uint32_t cnt = flac_count(a, u);
    if ((unsigned long long)f * FLAC_BLOCK >= cnt) return;
    const uint32_t n = min(FLAC_BLOCK, cnt - f * FLAC_BLOCK);
    const int16_t* src = a.slots + a.slot_off[u] + (unsigned long long)f * FLAC_BLOCK;
    for (uint32_t i = tid; i < n; i += FLAC_THREADS) sm.x[i] = src[i];
    __syncthreads();
    FlacFrame& d = a.frames[a.frame_base[u] + f];

    // CONSTANT when every sample equals the first
    int differs = 0;
    for (uint32_t i = tid; i < n; i += FLAC_THREADS) differs |= sm.x[i] != sm.x[0];
    differs = block_allreduce<FLAC_THREADS>(differs, OpMaxI32{}, reinterpret_cast<int*>(sm.red));
    uint8_t h[16];
    const uint32_t hdr = flac_frame_header(h, f, n, a.hz);
    if (!differs) {
        if (tid == 0) {
            d.bytes = hdr + 3 + 2;
            d.kind = FLAC_CONSTANT;
            d.order = 0;
            d.po = 0;
        }
        return;
    }

    // fixed order: the least sum of |residual| over samples 4 .. n-1 (the same range for every order), ties to the
    // lower order; order 0 for n <= 4.  Integer sums: order-free, so exact.
    const uint32_t i0 = tid * FLAC_PER_THREAD;
    uint32_t order = 0;
    if (n > 4) {
        unsigned long long e[5] = {0, 0, 0, 0, 0};
        for (uint32_t i = max(i0, 4u); i < min(i0 + FLAC_PER_THREAD, n); i++)
#pragma unroll
            for (int o = 0; o < 5; o++) e[o] += (unsigned long long)abs(flac_residual(sm.x, i, o));
        unsigned long long best = ~0ull;
        for (int o = 0; o < 5; o++) {
            const unsigned long long t = block_allreduce<FLAC_THREADS>(e[o], OpAddU64{}, sm.red);
            if (t < best) {
                best = t;
                order = o;
            }
        }
    }

    // zigzag residuals of that order, in place of the samples
    uint32_t zz[FLAC_PER_THREAD];
#pragma unroll
    for (int q = 0; q < FLAC_PER_THREAD; q++) {
        const uint32_t i = i0 + q;
        zz[q] = (i >= order && i < n) ? flac_zigzag(flac_residual(sm.x, i, order)) : 0u;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < FLAC_PER_THREAD; q++) sm.zz[i0 + q] = zz[q];

    // partition orders: po = 0 .. 8 while n % 2^po == 0 and (n >> po) > order.  Sums at the finest one, then up the tree.
    uint32_t po_f = 0;
    while (po_f < FLAC_MAX_PO && n % (2u << po_f) == 0 && (n >> (po_f + 1)) > order) po_f++;
    __syncthreads();
    {
        const uint32_t P = 1u << po_f, m = n >> po_f;
        for (uint32_t it = tid; it < P * (FLAC_KMAX + 1); it += FLAC_THREADS) {
            const uint32_t j = it / (FLAC_KMAX + 1), k = it % (FLAC_KMAX + 1);
            unsigned long long s = 0;
            for (uint32_t i = j ? j * m : order; i < (j + 1) * m; i++) s += sm.zz[i] >> k;
            sm.s[it] = s;
        }
    }
    __syncthreads();
    for (int po = (int)po_f; po >= 0; po--) {
        const uint32_t P = 1u << po, m = n >> po;
        unsigned long long bits = 0;
        if (tid < P) {
            const unsigned long long len = m - (tid ? 0 : order);
            unsigned long long best = ~0ull;
            uint32_t kb = 0;
            for (uint32_t k = 0; k <= FLAC_KMAX; k++) {
                const unsigned long long c = len * (k + 1) + sm.s[tid * (FLAC_KMAX + 1) + k];
                if (c < best) {
                    best = c;
                    kb = k;
                }
            }
            sm.kb[P - 1 + tid] = (uint8_t)kb;
            bits = 4 + best;
        }
        bits = block_allreduce<FLAC_THREADS>(bits, OpAddU64{}, sm.red);
        if (tid == 0) sm.level_bits[po] = bits;
        if (po) {   // merge pairs of partitions for the next coarser order
            unsigned long long v[FLAC_KMAX + 1];
            if (tid < P / 2)
#pragma unroll
                for (int k = 0; k <= FLAC_KMAX; k++)
                    v[k] = sm.s[(2 * tid) * (FLAC_KMAX + 1) + k] + sm.s[(2 * tid + 1) * (FLAC_KMAX + 1) + k];
            __syncthreads();
            if (tid < P / 2)
#pragma unroll
                for (int k = 0; k <= FLAC_KMAX; k++) sm.s[tid * (FLAC_KMAX + 1) + k] = v[k];
            __syncthreads();
        }
    }
    __syncthreads();
    uint32_t po = 0;
    for (uint32_t q = 1; q <= po_f; q++)
        if (sm.level_bits[q] < sm.level_bits[po]) po = q;
    const unsigned long long fixed_bits = 8ull + 16ull * order + 6ull + sm.level_bits[po];
    const unsigned long long verbatim_bits = 8ull + 16ull * n;
    const bool verbatim = verbatim_bits < fixed_bits;
    if (tid == 0) {
        d.kind = verbatim ? FLAC_VERBATIM : FLAC_FIXED;
        d.order = (uint8_t)order;
        d.po = (uint8_t)po;
        d.bytes = hdr + (uint32_t)(((verbatim ? verbatim_bits : fixed_bits) + 7) / 8) + 2;
    }
    if (!verbatim && tid < (1u << po)) d.k[tid] = sm.kb[(1u << po) - 1 + tid];
}

// ---------------------------------------------------------------- byte layout

__global__ void __launch_bounds__(1024) flac_scan_kernel(FlacArgs a, const uint32_t* __restrict__ err, uint32_t n, uint32_t* h_res) {
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0ull;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t u = base + (uint32_t)tid;
        unsigned long long v = 0;
        if (u < n) {
            const uint32_t frames = (flac_count(a, u) + FLAC_BLOCK - 1) / FLAC_BLOCK;
            FlacFrame* fr = a.frames + a.frame_base[u];
            uint32_t off = FLAC_HEADER_BYTES, lo = frames ? 0xffffffffu : 0u, hi = 0;
            for (uint32_t f = 0; f < frames; f++) {
                const uint32_t b = fr[f].bytes;
                fr[f].off = off;
                off += b;
                lo = min(lo, b);
                hi = max(hi, b);
            }
            a.uinfo[3 * u] = off;
            a.uinfo[3 * u + 1] = lo;
            a.uinfo[3 * u + 2] = hi;
            h_res[u] = a.counts[u];
            h_res[n + u] = err[u];
            h_res[2 * n + u] = off;
            v = ((unsigned long long)off + 15ull) & ~15ull;
        }
        unsigned long long inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) wsum[warp] = inc;
        __syncthreads();
        unsigned long long pre = s_carry;
        for (int w = 0; w < warp; w++) pre += wsum[w];
        if (u < n) a.byte_off[u] = pre + inc - v;
        __syncthreads();
        if (tid == 1023) s_carry = pre + inc;
        __syncthreads();
    }
    if (tid == 0) a.byte_off[n] = s_carry;
    __threadfence_system();
}

// ---------------------------------------------------------------- emission

constexpr uint32_t FLAC_WORDS = (FLAC_FRAME_MAX + 3) / 4;

// CRC-16 (0x8005, MSB first, init 0) is linear: crc(A || B) = crc(A) * x^(8 |B|) mod P  xor  crc(B).
__device__ __forceinline__ uint32_t crc16_mulmod(uint32_t a, uint32_t b) {
    uint32_t r = 0;
    for (int i = 15; i >= 0; i--) {
        r <<= 1;
        if (r & 0x10000u) r ^= 0x18005u;
        if ((b >> i) & 1u) r ^= a;
    }
    return r;
}
__device__ __forceinline__ uint32_t crc16_shift(uint32_t crc, uint32_t bytes) {   // crc * x^(8 bytes) mod P
    uint32_t base = 0x100u;   // x^8
    for (; bytes; bytes >>= 1) {
        if (bytes & 1u) crc = crc16_mulmod(crc, base);
        base = crc16_mulmod(base, base);
    }
    return crc;
}

struct FlacEmitSmem {
    int16_t x[FLAC_BLOCK];
    uint32_t w[FLAC_WORDS + 1];   // the frame, big-endian bit order inside every word
    uint16_t crc_table[256];
    uint32_t red[FLAC_THREADS / 32];
};

__device__ __forceinline__ void flac_put(uint32_t* w, uint32_t pos, uint32_t len, uint32_t v) {   // len <= 32
    if (!len) return;
    const unsigned long long x = (unsigned long long)v << (64 - (pos & 31) - len);
    atomicOr(w + (pos >> 5), (uint32_t)(x >> 32));
    if ((uint32_t)x) atomicOr(w + (pos >> 5) + 1, (uint32_t)x);
}
__device__ __forceinline__ uint32_t flac_byte(const uint32_t* w, uint32_t j) { return (w[j >> 2] >> (24 - 8 * (j & 3))) & 0xFFu; }

__global__ void __launch_bounds__(FLAC_THREADS) flac_emit_kernel(FlacArgs a, uint32_t u_base) {
    __shared__ FlacEmitSmem sm;
    const uint32_t u = u_base + blockIdx.y, f = blockIdx.x, tid = threadIdx.x;
    const uint32_t cnt = flac_count(a, u);
    uint8_t* file = a.out + a.byte_off[u];
    if (f == 0) {   // "fLaC" + STREAMINFO, and the zero padding up to the next 16-byte boundary
        const uint32_t bytes = a.uinfo[3 * u];
        if (tid < FLAC_HEADER_BYTES) {
            const uint32_t lo = a.uinfo[3 * u + 1], hi = a.uinfo[3 * u + 2];
            const unsigned long long pk = (unsigned long long)a.hz << 44 | 15ull << 36 | (unsigned long long)cnt;
            uint32_t b = 0;
            if (tid < 4) b = (uint8_t)"fLaC"[tid];
            else if (tid == 4) b = 0x80;   // last metadata block, type 0 (STREAMINFO)
            else if (tid == 7) b = 34;
            else if (tid == 8 || tid == 10) b = FLAC_BLOCK >> 8;
            else if (tid >= 12 && tid < 15) b = lo >> (8 * (14 - tid));
            else if (tid >= 15 && tid < 18) b = hi >> (8 * (17 - tid));
            else if (tid >= 18 && tid < 26) b = (uint32_t)(pk >> (8 * (25 - tid)));
            file[tid] = (uint8_t)b;
        }
        for (uint32_t j = bytes + tid; j < ((bytes + 15u) & ~15u); j += FLAC_THREADS) file[j] = 0;
    }
    if ((unsigned long long)f * FLAC_BLOCK >= cnt) return;
    const uint32_t n = min(FLAC_BLOCK, cnt - f * FLAC_BLOCK);
    const FlacFrame& d = a.frames[a.frame_base[u] + f];
    const int16_t* src = a.slots + a.slot_off[u] + (unsigned long long)f * FLAC_BLOCK;
    for (uint32_t i = tid; i < n; i += FLAC_THREADS) sm.x[i] = src[i];
    for (uint32_t i = tid; i <= FLAC_WORDS; i += FLAC_THREADS) sm.w[i] = 0;
    {
        uint32_t c = tid << 8;
        for (int b = 0; b < 8; b++) c = (c & 0x8000u) ? (c << 1) ^ 0x8005u : c << 1;
        sm.crc_table[tid] = (uint16_t)c;
    }
    __syncthreads();
    const uint32_t kind = d.kind, order = d.order, po = d.po, bytes = d.bytes;
    uint8_t h[16];
    const uint32_t hdr = flac_frame_header(h, f, n, a.hz);
    const uint32_t sb = 8 * hdr;   // subframe start (bits)
    if (tid == 0) {
        for (uint32_t i = 0; i < hdr; i++) flac_put(sm.w, 8 * i, 8, h[i]);
        flac_put(sm.w, sb, 8, kind == FLAC_CONSTANT ? 0u : kind == FLAC_VERBATIM ? 2u : (8u + order) << 1);
        if (kind == FLAC_CONSTANT) flac_put(sm.w, sb + 8, 16, (uint16_t)sm.x[0]);
        if (kind == FLAC_FIXED) flac_put(sm.w, sb + 8 + 16 * order, 6, po);   // method 00, partition order
    }
    const uint32_t i0 = tid * FLAC_PER_THREAD, i1 = min(i0 + FLAC_PER_THREAD, n);
    if (kind == FLAC_VERBATIM) {
        for (uint32_t i = i0; i < i1; i++) flac_put(sm.w, sb + 8 + 16 * i, 16, (uint16_t)sm.x[i]);
    } else if (kind == FLAC_FIXED) {
        const uint32_t m = n >> po;
        for (uint32_t i = i0; i < min(i1, order); i++) flac_put(sm.w, sb + 8 + 16 * i, 16, (uint16_t)sm.x[i]);
        // bit length of every residual code (with the 4-bit parameter in front of a partition's first one)
        uint32_t mine = 0;
        for (uint32_t i = max(i0, order); i < i1; i++) {
            const uint32_t j = i / m, k = d.k[j];
            mine += (flac_zigzag(flac_residual(sm.x, i, order)) >> k) + 1 + k + (i == (j ? j * m : order) ? 4 : 0);
        }
        uint32_t pos = block_excl_scan<FLAC_THREADS>(mine, OpAddU32{}, 0u, sm.red, false) + sb + 8 + 16 * order + 6;
        for (uint32_t i = max(i0, order); i < i1; i++) {
            const uint32_t j = i / m, k = d.k[j];
            if (i == (j ? j * m : order)) {
                flac_put(sm.w, pos, 4, k);
                pos += 4;
            }
            const uint32_t z = flac_zigzag(flac_residual(sm.x, i, order));
            pos += z >> k;   // the unary quotient's zeros
            flac_put(sm.w, pos, k + 1, (1u << k) | (z & ((1u << k) - 1u)));
            pos += k + 1;
        }
    }
    __syncthreads();
    // CRC-16 over bytes [0, bytes - 2): every thread one segment, shifted to the end and xor-ed together
    const uint32_t body = bytes - 2, seg = (body + FLAC_THREADS - 1) / FLAC_THREADS;
    const uint32_t b0 = min(body, tid * seg), b1 = min(body, b0 + seg);
    uint32_t crc = 0;
    for (uint32_t j = b0; j < b1; j++) crc = ((crc << 8) ^ sm.crc_table[((crc >> 8) ^ flac_byte(sm.w, j)) & 0xFFu]) & 0xFFFFu;
    crc = crc16_shift(crc, body - b1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, o);
    if ((tid & 31) == 0) sm.red[tid >> 5] = crc;
    __syncthreads();
    if (tid == 0) {
        uint32_t c = 0;
        for (int k = 0; k < FLAC_THREADS / 32; k++) c ^= sm.red[k];
        flac_put(sm.w, 8 * body, 16, c);
    }
    __syncthreads();
    uint8_t* dst = file + d.off;
    for (uint32_t j = tid; j < bytes; j += FLAC_THREADS) dst[j] = (uint8_t)flac_byte(sm.w, j);
}

}  // namespace ctts
