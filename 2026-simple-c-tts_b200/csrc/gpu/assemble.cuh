// assemble.cuh -- the persistent region-task kernel (see asm_common.cuh for the design).
#pragma once
#include "asm_common.cuh"
#include "asm_pitch.cuh"
#include "asm_unit.cuh"
#include "asm_word.cuh"

namespace ctts {

// ---------------------------------------------------------------- kernel

// apply_fade_out on the buffer tail (ctts.c:3028): `if (buf.count > 0) apply_fade_out(buf, count, a)`
__device__ void op_fade_out(State& s, const Smem& sm, const AsmArgs& A, uint32_t a) {
    if (a == 0) return;
    uint32_t f = a;
    if (s.cnt < a) {
        if (threadIdx.x == 0) sm.bcast[3] = 1u;   // the result depends on more than this task's ops (TASK_SOURCE)
        need_base(s, sm, A);
        const unsigned long long count = (unsigned long long)s.base + s.cnt;
        if (count == 0) return;
        if (count < f) f = (uint32_t)count;
        if (f > s.cnt && s.in_smem) enter_global(s, sm, A);
    }
    int16_t* p = s.w + ((int)s.cnt - (int)f);
    const float inv = 1.0f / (float)f;
    for (uint32_t i = threadIdx.x; i < f; i += ASM_THREADS)
        p[i] = f2s((float)p[i] * lut_lerp(A.tab.sine, (float)(f - i) * inv));
    __syncthreads();
}

// buffer_append_silence, ctts.c:3361
__device__ void op_silence(State& s, uint32_t n) {
    if ((unsigned long long)s.cnt + n > s.cap) { s.err = ERR_WINDOW_OVERFLOW; return; }
    int16_t* p = s.w + s.cnt;
    const int tid = threadIdx.x;
    // scalar head to the 16-byte grid, vector body, scalar tail
    uint32_t h = (8u - (uint32_t)((reinterpret_cast<uintptr_t>(p) >> 1) & 7u)) & 7u;
    if (h > n) h = n;
    if ((uint32_t)tid < h) p[tid] = 0;
    const uint32_t nv = (n - h) >> 3;
    int4* pv = reinterpret_cast<int4*>(p + h);
    for (uint32_t v = tid; v < nv; v += ASM_THREADS) pv[v] = make_int4(0, 0, 0, 0);
    const uint32_t t0 = h + (nv << 3);
    if (t0 + tid < n) p[t0 + tid] = 0;
    s.cnt += n;
    __syncthreads();
}

// The ticket thread 0 drew before this work item started: published in bcast[1] (read by everyone once the item is
// done), its descriptor copied into `next_task` behind the scenes.
__device__ __forceinline__ void fetch_next(const Smem& sm, const AsmArgs& A, RegionTask* next_task, uint32_t next_ticket) {
    const int tid = threadIdx.x;
    if (tid < 32) {
        const uint32_t n = __shfl_sync(0xffffffffu, next_ticket, 0);
        if (tid == 0) sm.bcast[1] = n;
        if (tid < 4 && n < A.n_tasks)
            cp_async16(reinterpret_cast<char*>(next_task) + 16 * tid, reinterpret_cast<const char*>(A.tasks + n) + 16 * tid);
    }
}

// CTTS_GPU_TASK_TIMES=1: CTA time per task class.  A development aid that costs 1.5 % when compiled in, so it is
// compiled OUT by default: build with CTTS_NVCC_EXTRA=-DCTTS_ASM_PROF=1 (see _build.py) to use it.
#ifndef CTTS_ASM_PROF
#define CTTS_ASM_PROF 0
#endif
__device__ __forceinline__ void task_time(const Smem& sm, const AsmArgs& A, int cls) {
    if (CTTS_ASM_PROF && A.prof && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        atomicAdd(A.prof + 2 * cls, (unsigned long long)((uint32_t)t - sm.bcast[5]));
        atomicAdd(A.prof + 2 * cls + 1, 1ull);
    }
}

// `task` lives in shared memory (fields are read where they are used: no registers held over the op loop); `next_ticket`
// is the ticket thread 0 drew before this task started: once the task's own first loads are on their way it is
// published in bcast[1] and its descriptor is copied into `next_task` behind the scenes.
__device__ __forceinline__ void run_task(const Smem& sm, const AsmArgs& A, uint32_t ti, const RegionTask& task, RegionTask* next_task,
                         uint32_t next_ticket) {
    const int tid = threadIdx.x;
    State s;
    s.dst = ((task.flags & TASK_TO_PRE) ? A.dst_pre : A.dst_final) + task.dst_off;
    s.dst_cap = task.dst_cap;
    s.cnt = 0;
    s.word_start = 0;
    s.err = 0;
    s.pred = task.pred;
    s.have_base = task.pred < 0;
    s.base = 0;
    s.in_smem = true;
    if (tid == 0) {
        sm.bcast[3] = 0u;                         // reached-back flag, read after the op loop: barriers in between
        if (CTTS_ASM_PROF && A.prof) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            sm.bcast[5] = (uint32_t)t;
        }
    }
    s.w = sm.win;
    s.cap = A.wcap;
    // ---- word-region deduplication.  What a word region holds right before its contour (units gathered, joined,
    // DC removed, crossfaded, pauses, trimming) depends on the ops of the region alone, as long as no count clamp
    // binds (the utterance is at least `thresh` samples long when the region starts) and nothing reaches back past the
    // region's start (the plan compiler proves that).  Equal regions of a batch are therefore computed ONCE per launch
    // -- the canonical tasks, first in ticket order, assembled as if the utterance were long -- and every other
    // occurrence copies the result and resumes at its own contour (whose factors differ from word to word).
    // Second level: tasks that are equal as a whole (same canonical region, same WORD_END bit for bit, nothing but
    // fade-outs / pauses / marks behind it).  The first of them in ticket order (TASK_SOURCE) stores what it flushes in
    // the region store too, the others (TASK_REUSE) copy that and run nothing.
    // Regions longer than the window (TASK_GLOBAL) take part as well: a canonical one is assembled in its region-store
    // slot, an occurrence copies the store straight into its utterance slot and resumes there, a source copies what it
    // appended to its slot into the store.
    // the task's ops, asynchronously (an op fetched from HBM per step would stall the whole CTA)
    {
        const uint32_t n_pref = min(task.op_end - task.op_begin, TASK_OPS_SMEM);
        if ((uint32_t)tid < 2 * n_pref) cp_async16(sm.ops + tid, reinterpret_cast<const int4*>(A.ops + task.op_begin) + tid);
    }
    const bool canon = (task.flags & TASK_CANON) != 0;
    uint32_t k_first = task.op_begin;
    bool resumed = false;
    if (canon) {
        s.dst = A.region_store + task.dst_off;
        s.have_base = true;
        s.base = CANON_BASE;
        if (task.flags & TASK_GLOBAL) {   // in place in the region store: nothing reaches back (the plan compiler proves it)
            s.in_smem = false;
            s.w = s.dst;
            s.cap = task.dst_cap;
        }
    } else if (task.region != NO_REGION) {
        // One round trip for everything this task waits for: lane 0 the predecessor's chain word, lane 1 the
        // canonical region's state, lane 2 the shared whole task's (their producers hold smaller tickets: running or
        // done).  bcast[0] = base, bcast[2] / bcast[4] = lengths (NO_REGION: the producer gave up on it).
        if (tid < 3) {
            const unsigned long long* p = nullptr;
            if (tid == 0 && !s.have_base && task.thresh != 0u) p = A.chain + s.pred;   // (threshold 0: the count is not needed yet)
            if (tid == 1) p = A.region_state + task.region;
            if (tid == 2 && (task.flags & TASK_REUSE)) p = A.region_state + task.whole;
            unsigned long long v = NO_REGION;
            if (p) {
                unsigned ns = 20;
                while ((uint32_t)((v = ld_acquire_u64(p)) >> 32) != A.epoch) {
                    __nanosleep(ns);
                    if (ns < 640) ns *= 2;
                }
            }
            sm.bcast[2 * tid] = (uint32_t)v;
        }
        __syncthreads();
        if (!s.have_base && task.thresh != 0u) {
            s.base = sm.bcast[0];
            s.have_base = true;
        }
        if (s.base >= task.thresh) {
            const uint32_t len_whole = sm.bcast[4], len_region = sm.bcast[2];
            const uint32_t cap = (task.flags & TASK_GLOBAL) ? NO_REGION : s.cap;   // TASK_GLOBAL: the slot's, checked below
            uint32_t len = NO_REGION;
            unsigned long long at = 0;
            if (len_whole != NO_REGION && len_whole <= cap) {
                len = len_whole;
                at = 8ull * task.whole_at;
                k_first = task.op_end;
            } else if (len_region != NO_REGION && len_region <= cap) {
                len = len_region;
                at = 8ull * task.region_at;
                k_first = task.w_op;
                resumed = true;
            }
            if (len != NO_REGION) {
                s.cnt = len;
                if (!(task.flags & TASK_GLOBAL)) {   // region store -> window (written by another CTA during this launch: L2, not the read-only path)
                    const int4* src = reinterpret_cast<const int4*>(A.region_store + at);
                    int4* dstw = reinterpret_cast<int4*>(sm.win);
                    for (uint32_t v = tid; v < (len + 7) >> 3; v += ASM_THREADS) cp_async16(dstw + v, src + v);
                }
            }
        }
    }
    if ((task.flags & TASK_GLOBAL) && !canon) {
        // the region does not fit the shared window: assemble it in place in the HBM slot
        need_base(s, sm, A);
        s.in_smem = false;
        s.w = s.dst + s.base;
        s.cap = s.dst_cap > s.base ? s.dst_cap - s.base : 0u;
        if (s.cnt > s.cap) {   // the stored samples do not fit the slot: assemble them, and fail, as without the store
            s.cnt = 0;
            k_first = task.op_begin;
            resumed = false;
        } else if (k_first != task.op_begin) {
            copy_from_store(s.w, A.region_store + 8ull * (resumed ? task.region_at : task.whole_at), s.cnt);
        }
        __threadfence();
    }
    cp_async_wait_all();
    __syncthreads();
    fetch_next(sm, A, next_task, next_ticket);
    for (uint32_t k = k_first; k < task.op_end && !s.err; k++) {
        ctts_plan_op op;
        {
            const uint32_t rel = k - task.op_begin;
            int4 lo, hi;
            if (rel < TASK_OPS_SMEM) {
                lo = sm.ops[2 * rel];
                hi = sm.ops[2 * rel + 1];
            } else {
                const int4* p = reinterpret_cast<const int4*>(A.ops + k);
                lo = __ldg(p);
                hi = __ldg(p + 1);
            }
            *reinterpret_cast<int4*>(&op) = lo;
            *(reinterpret_cast<int4*>(&op) + 1) = hi;
        }
        switch (op.kind) {
            case OP_NOP:
                break;
            case CTTS_OP_UNIT:
                op_unit(s, sm, A, op);
                break;
            case CTTS_OP_SILENCE:
                op_silence(s, op.a);
                break;
            case CTTS_OP_FADE_OUT:
                op_fade_out(s, sm, A, op.a);
                break;
            case CTTS_OP_WORD_END: {
                unsigned long long t0 = 0;
                const bool timed = CTTS_ASM_PROF && A.prof && !s.in_smem;
                if (timed && tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
                if (canon) op_word_end(s, sm, A, task.big, op, true, false);              // stops in front of the contour
                else op_word_end(s, sm, A, task.big, op, !(resumed && k == task.w_op), true);
                if (timed && tid == 0) {
                    unsigned long long t1;
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    atomicAdd(A.prof + 10, t1 - t0);
                    atomicAdd(A.prof + 11, 1ull);
                }
                break;
            }
            case CTTS_OP_MARK:   // word_start_sample = buf.count, ctts.c:3723, :3765
                s.word_start = s.cnt;
                break;
            default:
                s.err = ERR_BAD_OP;
        }
    }

    if (canon) {
        // ---- the canonical region goes to the region store (TASK_GLOBAL: it is there already); a region that left
        //      the window (cannot happen for regions the plan compiler accepts) or failed is marked unusable: its
        //      occurrences assemble themselves
        const bool ok = !s.err && s.in_smem == !(task.flags & TASK_GLOBAL) && s.cnt <= task.dst_cap;
        if (ok && s.in_smem) {
            const int4* srcw = reinterpret_cast<const int4*>(sm.win);
            int4* d = reinterpret_cast<int4*>(s.dst);
            for (uint32_t v = tid; v < (s.cnt + 7) >> 3; v += ASM_THREADS) d[v] = srcw[v];
        }
        __syncthreads();
        if (tid == 0) st_release_u64(A.region_state + task.region, ((unsigned long long)A.epoch << 32) | (ok ? s.cnt : NO_REGION));
        task_time(sm, A, 0);
        return;
    }
    if (task.flags & TASK_SOURCE) {
        // ---- what this task appends goes to the region store as well, unless it depends on more than the task's ops
        //      (TASK_GLOBAL: from the utterance slot, where it was appended)
        const bool global = (task.flags & TASK_GLOBAL) != 0;
        const bool ok = resumed && sm.bcast[3] == 0u && !s.err && s.in_smem == !global && s.cnt <= task.bound;
        if (ok && global) {
            __syncthreads();   // every thread's last samples are in the slot
            copy_to_store(A.region_store + 8ull * task.whole_at, s.dst + s.base, s.cnt);
        } else if (ok) {
            const int4* srcw = reinterpret_cast<const int4*>(sm.win);
            int4* d = reinterpret_cast<int4*>(A.region_store + 8ull * task.whole_at);
            for (uint32_t v = tid; v < (s.cnt + 7) >> 3; v += ASM_THREADS) d[v] = srcw[v];
        }
        __syncthreads();   // the CTA's stores happen before thread 0's release (barrier), the release is cumulative
        if (tid == 0) st_release_u64(A.region_state + task.whole, ((unsigned long long)A.epoch << 32) | (ok ? s.cnt : NO_REGION));
    }
    // ---- publish: the region's final position is base, known from the predecessor
    need_base(s, sm, A);
    __syncthreads();
    if (s.in_smem) {
        if ((unsigned long long)s.base + s.cnt > s.dst_cap) s.err = s.err ? s.err : ERR_SLOT_OVERFLOW;
        else flush_window(s, sm, 0, s.cnt);
    }
    __syncthreads();
    if (tid == 0) {
        const uint32_t total = s.base + s.cnt;
        if (s.err) atomicMax(A.err + task.utt, s.err);
        if (task.flags & TASK_LAST) {
            if (task.flags & TASK_TO_PRE) A.pre_counts[task.utt] = total;
            else A.out_counts[task.utt] = total;
        }
        st_release_u64(A.chain + ti, ((unsigned long long)A.epoch << 32) | total);
    }
    task_time(sm, A, k_first == task.op_end && task.op_end != task.op_begin ? 1 : resumed ? 2 : (task.flags & TASK_GLOBAL) || !s.in_smem ? 4 : 3);
}

__global__ void __launch_bounds__(ASM_THREADS, 3) assemble_kernel(const AsmArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // fixed-size parts first: their addresses are compile-time offsets (see SMEM_* in asm_common.cuh)
    Smem sm;
    sm.hann256 = reinterpret_cast<float*>(smem_raw + SMEM_HANN);
    sm.nrm2 = reinterpret_cast<float*>(smem_raw + SMEM_NRM2);
    sm.red = reinterpret_cast<unsigned long long*>(smem_raw + SMEM_RED);
    sm.bcast = reinterpret_cast<uint32_t*>(smem_raw + SMEM_BCAST);
    sm.ops = reinterpret_cast<int4*>(smem_raw + SMEM_OPS);
    sm.scratch = reinterpret_cast<uint32_t*>(smem_raw + SMEM_SCRATCH);
    sm.hstage = reinterpret_cast<int16_t*>(smem_raw + SMEM_HSTAGE);
    sm.win = sm.hstage + A.hcap;

    const int tid = threadIdx.x;
    for (int i = tid; i < PITCH_FRAME; i += ASM_THREADS) sm.hann256[i] = __ldg(A.tab.hann256 + i);
    // norm of a sample covered by two frames: (0 + w[i+128]) + w[i], the reference's accumulation order
    for (int i = tid; i < PITCH_FRAME / 2; i += ASM_THREADS)
        sm.nrm2[i] = __ldg(A.tab.hann256 + i + PITCH_FRAME / 2) + __ldg(A.tab.hann256 + i);
    __syncthreads();

    // persistent CTAs: tasks are taken in ticket order (see the header comment), one ticket AHEAD: the atomic and the
    // descriptor fetch of the next task overlap the running one.  (Still deadlock-free: the smallest unfinished
    // ticket is always running -- its holder has no smaller ticket left.)
    RegionTask* tbuf = reinterpret_cast<RegionTask*>(smem_raw + SMEM_TASK);
    if (tid == 0) sm.bcast[1] = atomicAdd(A.ticket, 1u);
    __syncthreads();
    uint32_t ti = sm.bcast[1];
    if (tid < 4 && ti < A.n_tasks)
        cp_async16(reinterpret_cast<char*>(tbuf) + 16 * tid, reinterpret_cast<const char*>(A.tasks + ti) + 16 * tid);
    uint32_t buf = 0;
    while (ti < A.n_tasks) {
        uint32_t next_ticket = 0;
        if (tid == 0) next_ticket = atomicAdd(A.ticket, 1u);   // consumed inside run_task, a few loads later
        cp_async_wait_all();
        __syncthreads();
        run_task(sm, A, ti, tbuf[buf], tbuf + (buf ^ 1u), next_ticket);
        __syncthreads();
        ti = sm.bcast[1];
        buf ^= 1u;
    }
}

// ---------------------------------------------------------------- packed output (device prefix sum + gather)

// Utterance slots are spaced by host-known upper bounds; what the caller wants are the samples that exist.
// pack_scan_kernel: exclusive prefix sum of the counts rounded up to 8 samples (every utterance starts on a
// 16-byte boundary) -> pack_off[0..n].  One CTA.  It also stores counts and error flags straight into
// page-locked host memory (h_res: counts [n], flags [n]): the host needs them to size the PCM copy, and a
// device->host copy of them would queue behind the PCM of earlier pieces on the copy engine.
constexpr int PACK_THREADS = 256;
__global__ void __launch_bounds__(1024) pack_scan_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ err, uint32_t n,
                                                         unsigned long long* __restrict__ pack_off, uint32_t* h_res) {
    __shared__ unsigned long long wsum[32];
    __shared__ unsigned long long s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0ull;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t u = base + (uint32_t)tid;
        const unsigned long long v = u < n ? (((unsigned long long)counts[u] + 7ull) & ~7ull) : 0ull;
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
        if (u < n) {
            pack_off[u] = pre + inc - v;
            h_res[u] = counts[u];
            h_res[n + u] = err[u];
        }
        __syncthreads();
        if (tid == 1023) s_carry = pre + inc;
        __syncthreads();
    }
    if (tid == 0) pack_off[n] = s_carry;
    __threadfence_system();
}

// pack_copy_kernel: utterance blockIdx.y, tile blockIdx.x of 8 * PACK_THREADS * 4 samples: slot -> packed
// position, 16-byte vectors (both sides are 16-byte aligned); the <= 7 samples of padding are written as zeros.
constexpr uint32_t PACK_TILE = 8u * PACK_THREADS * 4u;
__global__ void __launch_bounds__(PACK_THREADS) pack_copy_kernel(const int16_t* __restrict__ slots, const unsigned long long* __restrict__ slot_off,
                                                                 const uint32_t* __restrict__ counts, const unsigned long long* __restrict__ pack_off,
                                                                 int16_t* __restrict__ packed) {
    const uint32_t u = blockIdx.y;
    const uint32_t cnt = counts[u];
    const uint32_t t0 = blockIdx.x * PACK_TILE;
    if (t0 >= cnt) return;
    const int4* src = reinterpret_cast<const int4*>(slots + slot_off[u]);
    int4* dst = reinterpret_cast<int4*>(packed + pack_off[u]);
    const uint32_t nvec = (cnt + 7u) >> 3;
    const uint32_t v1 = min(nvec, (t0 + PACK_TILE) >> 3);
    for (uint32_t v = (t0 >> 3) + threadIdx.x; v < v1; v += PACK_THREADS) {
        int4 q = __ldcs(src + v);
        if (8u * v + 8u > cnt) {   // the last vector: zero the padding
            int16_t* e = reinterpret_cast<int16_t*>(&q);
#pragma unroll
            for (int k = 0; k < 8; k++)
                if (8u * v + (uint32_t)k >= cnt) e[k] = 0;
        }
        __stcs(dst + v, q);
    }
}

}  // namespace ctts
