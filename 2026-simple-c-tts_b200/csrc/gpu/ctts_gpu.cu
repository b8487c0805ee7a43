// ctts_gpu.cu -- C-ABI (include/ctts_gpu.h) over the sm_100a kernels.
//
// Host side only does plumbing: parse voice.db, re-pack and upload the PCM
// pool and tables, turn a CSR plan into per-utterance tasks and an output
// layout, launch kernels on one stream.  There is no CPU implementation of any
// sample operation in this library.
#include "ctts_gpu.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <numeric>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "assemble.cuh"
#include "wsola.cuh"
#include "resample.cuh"
#include "flac.cuh"
#include "g711.cuh"
#include "loudness.cuh"

extern "C" void ctts_host_tables(float* fade_out, float* fade_in, float* sine, float* hann256,
                                 float* hann512);
extern "C" void ctts_host_resample_taps(unsigned L, unsigned M, float* g);
extern "C" void ctts_host_loudness_filter(unsigned fs, double* shelf, double* hp);
extern "C" void ctts_host_loudness_gains(unsigned* table);
extern "C" unsigned ctts_host_loudness_ceiling(float ceiling_dbfs);
extern "C" void ctts_host_true_peak_taps(float* h);

// Launch geometry of resample_kernel for the reduced ratio L/M (host only, no CUDA call; tests restate the kernel's
// tile arithmetic against it): kp taps per phase row (a multiple of 4), the filter delay c, the staging bound
// smem_floats of one tile, and the tiles (grid.x) that cover every output of an utterance of at most max_out
// output samples.
extern "C" void ctts_host_resample_geometry(uint32_t L, uint32_t M, uint64_t max_out, uint32_t* kp, uint32_t* c,
                                            uint32_t* smem_floats, uint32_t* tiles) {
    const uint32_t R = std::max(L, M), N = 2u * 40u * R + 1u;
    *kp = ((N + L - 1) / L + 3) & ~3u;
    *c = 40u * R;
    // input span of a tile of RS_THREADS work items: they cover at most d + 1 rows of L * RS_COPIES outputs
    const uint64_t d = (uint64_t)(L - 1 + ctts::RS_THREADS - 1) / L;
    const uint64_t out_span = d * L * ctts::RS_COPIES + (uint64_t)L * ctts::RS_COPIES;
    *smem_floats = (uint32_t)(((out_span * M) / L + 2 + *kp + 3) & ~3ull);
    const uint64_t row = (uint64_t)L * ctts::RS_COPIES;
    *tiles = (uint32_t)std::max<uint64_t>(((max_out + row - 1) / row * L + ctts::RS_THREADS - 1) / ctts::RS_THREADS, 1);
}

namespace {

struct DbHeader {  // ctts.h:84-98
    uint32_t magic, version, unit_count, sample_rate, bits_per_sample, index_offset, strings_offset,
        audio_offset, total_samples, max_unit_chars, hash_table_size, hash_table_offset;
    uint8_t reserved[16];
};
struct DbEntry {  // ctts.h:101-111
    uint32_t hash, string_offset;
    uint16_t string_len, char_count;
    uint32_t audio_offset, sample_count, flags, next_hash, reserved;
};
static_assert(sizeof(DbHeader) == 64 && sizeof(DbEntry) == 32, "voice.db records");
static_assert(sizeof(ctts_plan_op) == 32, "plan op");

inline uint64_t up8(uint64_t v) { return (v + 7) & ~7ull; }

}  // namespace

// Development / test knobs, read from the environment ONCE, by ctts_gpu_init (never on the call path).
struct Knobs {
    bool trace = false;               // CTTS_GPU_TRACE: timing lines on stderr
    int host_threads = 0;             // CTTS_GPU_HOST_THREADS: threads of the plan scan (0: default 4)
    int pitch_slots = 0;              // CTTS_GPU_PITCH_SLOTS: capacity of the unit-head pitch table (tests: a table that fills up)
    int ctas_per_sm = 3;              // CTTS_GPU_CTAS_PER_SM: occupancy the assembly window is sized for
    int window = 0;                   // CTTS_GPU_WINDOW: shared window in samples (tests: force the HBM-window path)
    uint64_t piece_samples = 192ull << 20;   // CTTS_GPU_CHUNK_SAMPLES: size of the pieces of the three batch calls (slot samples; packed: / 2800 ops)
    bool task_times = false;          // CTTS_GPU_TASK_TIMES=1: resident plans print the time their CTAs spent per task class
                                      // (only in a library built with -DCTTS_ASM_PROF=1)
    int region_dedup = 2;             // CTTS_GPU_REGION_DEDUP=0: assemble every word region of a batch, equal ones too;
                                      // 1: share equal regions up to their contour; 2: equal whole tasks as well
    bool wsola_speculate = true;      // CTTS_GPU_WSOLA_SPECULATE=0: walk every WSOLA chain frame by frame
    uint32_t wsola_force_bad = 0;     // CTTS_GPU_WSOLA_FORCE_BAD=N: report every N-th frame as unverified (tests of the repair path)

    void read_env() {
        auto num = [](const char* name, long long dflt) {
            const char* e = getenv(name);
            return e && *e ? strtoll(e, nullptr, 10) : dflt;
        };
        trace = getenv("CTTS_GPU_TRACE") != nullptr;
        host_threads = (int)std::max(0ll, std::min(16ll, num("CTTS_GPU_HOST_THREADS", 0)));
        pitch_slots = (int)std::max(0ll, num("CTTS_GPU_PITCH_SLOTS", 0));
        ctas_per_sm = (int)std::max(1ll, std::min(8ll, num("CTTS_GPU_CTAS_PER_SM", 3)));
        window = (int)std::max(0ll, num("CTTS_GPU_WINDOW", 0));
        piece_samples = (uint64_t)std::max(1ll, num("CTTS_GPU_CHUNK_SAMPLES", 192ll << 20));
        region_dedup = (int)num("CTTS_GPU_REGION_DEDUP", 2);
        task_times = num("CTTS_GPU_TASK_TIMES", 0) != 0;
        wsola_speculate = num("CTTS_GPU_WSOLA_SPECULATE", 1) != 0;
        wsola_force_bad = (uint32_t)std::max(0ll, num("CTTS_GPU_WSOLA_FORCE_BAD", 0));
    }
};

struct Arena {
    char* d = nullptr;
    size_t d_cap = 0;
    char* h = nullptr;   // pinned
    size_t h_cap = 0;
};

struct ctts_gpu_plan;
struct ctts_gpu_session;

struct ctts_gpu_ctx {
    int device = 0;
    Knobs knobs;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    int16_t* d_pool = nullptr;
    uint32_t* d_unit_off = nullptr;
    uint32_t* d_unit_cnt = nullptr;
    float* d_tables = nullptr;  // fade_out, fade_in, sine (1024 each), hann256, hann512, xfade4 (4096)
    // normalize_rms applied to every unit, once per target_rms this context has seen
    // (normalize_pool_kernel); plans keep pointers into these, they live as long as the context
    struct NormPool {
        float target_rms = 0;
        int16_t* d_pool = nullptr;
        int4* d_meta = nullptr;
        // estimate_pitch of a unit's (normalized, untouched) head over R samples: table slots,
        // filled by unit_pitch_kernel when the plan compiler first meets a (unit, R) pair
        float* d_pitch = nullptr;
        uint32_t pitch_cap = 0, pitch_used = 0;
        std::vector<std::vector<std::pair<uint32_t, uint32_t>>> pitch_slots;   // per unit: (R, slot)
    };
    std::vector<NormPool*> norm_pools;
    // output-rate conversion (DESIGN.md 3.4): one tap table per rate this context has seen; plans keep a
    // pointer to the one they were created under, so tables live as long as the context
    struct RsTable {
        uint32_t hz = 0, L = 1, M = 1;
        uint32_t kp = 0;            // taps per phase row (multiple of 4)
        uint32_t c = 0;             // H * R: the filter's centre
        uint32_t smem_floats = 0;   // bound on the input span of one resample_kernel tile
        float* d_taps = nullptr;    // L rows of kp
    };
    std::vector<RsTable*> rs_tables;
    RsTable* rs = nullptr;          // the output rate of the context; nullptr: the native 22 050 Hz
    int rs_smem_attr = 48 * 1024;   // dynamic shared memory resample_kernel may use on this device
    // loudness normalization (DESIGN.md 3.6): one setting per (output rate, target, ceiling) this context has seen;
    // plans keep a pointer to the one they were created under
    struct LdTable {
        uint32_t hz = 0;
        float target = 0, ceiling = 0;
        bool true_peak = false;     // the ceiling holds the true (4x oversampled) peak, not the sample peak
        uint32_t ceiling_q = 0;     // A
        ctts::LdFilter f{};         // the K-weighting at hz and its transitions (kernel parameters)
        float tp_h[3][12] = {};     // true_peak: the interpolator's phases 1 .. 3 as LdArgs::tp_h lays them out
    };
    std::vector<LdTable*> ld_tables;
    LdTable* ld = nullptr;          // nullptr: the stage is off
    uint32_t* d_ld_gains = nullptr; // the gain table, uploaded by the first ctts_gpu_set_loudness that turns the stage on
    uint64_t pool_samples = 0;
    uint32_t n_units = 0;
    uint32_t max_unit = 0;
    std::vector<uint32_t> unit_cnt;
    std::vector<uint32_t> unit_off;   // offsets into the re-packed pool (samples, multiples of 8)
    int sm_count = 0;
    int smem_per_sm = 0;
    int smem_optin = 0;
    // A batch is worked on in PIECES (contiguous utterance ranges); up to kLanes (4) pieces are in flight: the
    // host compiles piece c+1 while the device assembles piece c and piece c-1 is copied to the caller.
    // Every lane owns grow-only workspaces (no cudaMalloc / cudaFree per call); device capacities count bytes.
    static constexpr int kLanes = 4;
    struct Lane {
        Arena arena;                       // device workspace + pinned staging of the plan upload
        int16_t* d_out = nullptr;          // the piece's output slots (native rate: where the kernels write)
        uint64_t d_out_cap = 0;
        int16_t* d_rs = nullptr;           // output-rate slots (only when the context converts the rate)
        uint64_t d_rs_cap = 0;
        uint8_t* d_pack = nullptr;         // packed mode: the utterances back to back (PCM samples, G.711 codes or FLAC files)
        uint64_t d_pack_cap = 0;
        unsigned long long* d_pack_off = nullptr;   // packed mode: ResLayout
        uint64_t d_pack_off_cap = 0;
        ctts::FlacFrame* d_frames = nullptr;   // FLAC sessions: one descriptor per frame a slot can hold
        uint64_t d_frames_cap = 0;
        uint32_t* d_flac_info = nullptr;   // FLAC sessions: per utterance file bytes, min and max frame bytes
        uint64_t d_flac_info_cap = 0;
        uint32_t* h_res = nullptr;         // pinned: ResLayout
        size_t h_res_cap = 0;              // in 4-byte words
        cudaEvent_t kernels_done = nullptr, counts_ready = nullptr, copied = nullptr;
        ctts_gpu_plan* plan = nullptr;     // piece in flight
        uint32_t* user_counts = nullptr;   // where its counts go
        uint64_t* user_offsets = nullptr;  // packed mode: where its offsets go
        uint32_t* user_bytes = nullptr;    // FLAC sessions: where its file sizes go
        bool copy_pending = false;         // packed mode: the PCM copy is enqueued once the counts are on the host
        uint32_t utt_base = 0, n = 0;      // its utterances in the session's numbering
        bool busy = false;
    };
    Lane lane[kLanes];
    cudaStream_t copy_stream = nullptr;
    ctts_gpu_session* session = nullptr;   // at most one at a time
    char err[512] = {0};
};

struct ctts_gpu_plan {
    ctts_gpu_ctx* ctx = nullptr;
    uint32_t n_utts = 0;
    ctts_assembly_params prm{};
    std::vector<uint64_t> offsets;  // n_utts + 1, output-rate slots (what callers see)
    std::vector<uint64_t> bounds;   // output-rate bounds
    ctts_gpu_ctx::RsTable* rs = nullptr;   // rate conversion the plan was created under (nullptr: native rate)
    std::vector<uint64_t> n_offsets;       // native-rate slots, where the assembly and WSOLA kernels write (== offsets without rs)
    // the plan's offset table: (rs: native slot offsets [n + 1],) output-rate slot offsets [n + 1], (ld: the first
    // chunk of every utterance [n + 1], ld->true_peak: its first ld_true_peak_kernel tile [n + 1]); slot_off() is
    // the output-rate section
    unsigned long long* d_off = nullptr;
    uint32_t* d_rs_counts = nullptr;       // rs: output-rate counts
    uint32_t* d_final_counts = nullptr;    // the counts callers see: d_rs_counts with rs, else d_counts
    uint32_t rs_tiles = 0;                 // rs: grid.x of resample_kernel
    int16_t* d_nat_owned = nullptr;        // resident plan with rs: its native slots
    const ctts_gpu_ctx::LdTable* ld = nullptr;   // loudness setting the plan was created under (nullptr: off)
    double* d_ld_state = nullptr;                // ld: 4 per chunk
    double* d_ld_energy = nullptr;               // ld: per chunk
    uint32_t* d_ld_peak = nullptr;               // ld: per chunk
    double* d_ld_lufs = nullptr;                 // ld: per utterance
    uint32_t* d_ld_gain = nullptr;               // ld: per utterance
    uint32_t ld_tiles = 0, ld_apply_tiles = 0;   // ld: grid.x of the chunk passes and of ld_apply_kernel
    float* d_ld_tp_tile = nullptr;               // ld->true_peak: per (utterance, tile) of ld_true_peak_kernel
    float* d_ld_tp = nullptr;                    // ld->true_peak: P per utterance
    uint32_t ld_tp_tiles = 0;                    // ld->true_peak: grid.x of ld_true_peak_kernel
    Arena* arena = nullptr;         // device buffers live in a lane's arena (batch path); else cudaMalloc'ed
    uint32_t op0 = 0;               // first op of the plan's utterances in the caller's op array (ops are kept from there on)
    std::vector<void*> owned;       // else: cudaMalloc'ed buffers to free
    ctts_gpu_ctx::NormPool* np = nullptr;   // context-owned: normalized pool and its tables
    ctts_plan_op* d_ops = nullptr;
    ctts::RegionTask* d_tasks = nullptr;
    unsigned long long* d_chain = nullptr;
    uint32_t* d_ticket = nullptr;
    unsigned long long* d_prof = nullptr;   // CTTS_GPU_TASK_TIMES: per task class {ns, tasks}
    int16_t* d_region_store = nullptr;              // canonical word regions (see run_task in assemble.cuh)
    unsigned long long* d_region_state = nullptr;
    size_t d_used = 0;              // arena mode: device bytes taken by prepare_plan (build_tasks continues from here)
    uint32_t n_tasks = 0;
    uint32_t grid = 0;              // CTAs of assemble_kernel
    uint32_t epoch = 0;
    ctts::StretchTask* d_stasks = nullptr;
    uint32_t* d_counts = nullptr;
    uint32_t* d_pre_counts = nullptr;
    uint32_t* d_err = nullptr;
    uint32_t* d_trim = nullptr;
    uint32_t trim_words = 0;
    int16_t* d_pre = nullptr;
    uint32_t* d_frame_pos = nullptr;
    uint32_t* d_n_frames = nullptr;
    uint32_t* d_ola_task = nullptr;
    uint32_t* d_ola_first = nullptr;
    uint32_t n_stretch = 0;
    uint32_t n_ola_blocks = 0;
    uint32_t verify_tiles = 0;      // tiles of the longest stretched utterance (grid.x of wsola_verify_kernel)
    int16_t* d_out_owned = nullptr;
    int16_t* d_out_last = nullptr;
    std::vector<uint64_t> pre_off;   // per utterance (stretch only), else ~0
    std::vector<uint64_t> pre_cap;
    uint32_t wcap = 0, hcap = 0, smem_bytes = 0;
    ctts_gpu_run_info info{};
    // builder state (prepare_plan -> build_tasks)
    ctts_plan_op* h_ops = nullptr;          // staging: pinned (lane arena) or h_staging
    ctts::RegionTask* h_tasks = nullptr;
    std::vector<char> h_staging;            // resident plans: pageable staging of the uploads, freed by build_tasks
    uint32_t n_big = 0, big_cap = 0, occ = 1;
};

namespace {

// why the last ctts_gpu_init of this thread failed (there is no context to hold the text then):
// ctts_gpu_last_error(NULL) returns it
thread_local char g_init_err[512] = "no context";

int fail(ctts_gpu_ctx* c, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    if (c) vsnprintf(c->err, sizeof c->err, fmt, ap);
    else vsnprintf(g_init_err, sizeof g_init_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CU(ctx, call)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail((ctx), CTTS_GPU_ERR_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                   \
    } while (0)

// speed handling of ctts_synthesize / time_stretch (ctts.c:3907, :3493-3503):
// returns true when the utterance goes through WSOLA and sets the synthesis hop
bool needs_stretch(float speed, uint32_t* hop) {
    if (speed == 1.0f) return false;
    if (speed < 0.5f) speed = 0.5f;
    if (speed > 2.0f) speed = 2.0f;
    if (fabsf(speed - 1.0f) < 0.01f) return false;  // plain copy
    size_t h = (size_t)((float)(size_t)128 / speed);
    if (h < 1) h = 1;
    *hop = (uint32_t)h;
    return true;
}

uint64_t stretch_bound(uint64_t pre, uint32_t hop) {
    uint64_t frames = pre > 512 ? (pre - 512) / 128 + 1 : 1;
    return frames * hop + 512;
}

// samples at the output rate of n native samples: ceil(n * L / M)
uint64_t rate_bound(const ctts_gpu_ctx::RsTable* rs, uint64_t n) { return rs ? (n * rs->L + rs->M - 1) / rs->M : n; }

// the output-rate slot offsets in the plan's offset table
unsigned long long* slot_off(const ctts_gpu_plan* p) { return p->d_off + (p->rs ? (size_t)p->n_utts + 1 : 0); }

// Upper bound of the samples a UNIT op appends, given a lower bound L of the samples already in
// the current region.  The crossfade consumes a = min(xf, count, n) samples of the tail
// (ctts.c:3319-3321) and count >= L, so a >= min(xf, n, L) whenever the unit is certain to be
// joined (not after a word boundary and the buffer is certainly not empty).  L is updated to a
// lower bound of the region length after the append (count + n - a >= max(L + n - min(xf, n), n)).
inline uint64_t unit_append_bound(const ctts_plan_op& op, uint32_t n, uint64_t& L) {
    if (n == 0) return 0;
    const bool boundary = (op.flags & CTTS_UNIT_AFTER_BOUNDARY) != 0;
    if (boundary) {
        L += n;
        return n;
    }
    const uint64_t m = std::min<uint64_t>(op.b, n);
    if (L == 0) {   // joined or not: decided on the device
        L = n;
        return n;
    }
    const uint64_t a_lb = std::min<uint64_t>(m, L);
    L = std::max<uint64_t>(L + n - m, n);
    return n - a_lb;
}

struct PlanScan {
    std::vector<uint64_t> pre, bound;   // per utterance: pre-stretch / output upper bounds
    uint32_t xf_max = 0;
    uint64_t region_max = 0, n_regions = 0, n_big_regions = 0, big_region_max = 0;
    bool bad_factor = false, any_stretch = false;
};

// pass A over the plan: validation, upper bounds, global maxima
// (utterances [u0, u1); pre / bound are written through `sc`, the scalars into `sc` too)
int scan_range(const ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, uint64_t big_threshold, PlanScan* sc, uint32_t* bad_utt,
               uint32_t u0, uint32_t u1, uint64_t* pre_out, uint64_t* bound_out) {
    const std::vector<uint32_t>& ucnt = ctx->unit_cnt;
    for (uint32_t u = u0; u < u1; u++) {
        const uint32_t b = plan->utt_op_begin[u], e = plan->utt_op_begin[u + 1];
        *bad_utt = u;
        if (b > e || e > plan->n_ops) return CTTS_GPU_ERR_INVALID_ARG;
        uint64_t total = 0, cur = 0, L = 0;
        auto close_region = [&] {
            total += cur;
            if (cur > sc->region_max) sc->region_max = cur;
            if (cur > big_threshold) {
                sc->n_big_regions++;
                if (cur > sc->big_region_max) sc->big_region_max = cur;
            }
            cur = 0;
            L = 0;
            sc->n_regions++;
        };
        for (uint32_t k = b; k < e; k++) {
            const ctts_plan_op& op = plan->ops[k];
            switch (op.kind) {
                case CTTS_OP_UNIT:
                    if (op.a >= ctx->n_units) return CTTS_GPU_ERR_INVALID_ARG;
                    cur += unit_append_bound(op, ucnt[op.a], L);
                    if (op.b > sc->xf_max) sc->xf_max = op.b;
                    break;
                case CTTS_OP_SILENCE:
                    cur += op.a;
                    L += op.a;
                    break;
                case CTTS_OP_FADE_OUT:
                    break;
                case CTTS_OP_WORD_END:
                    if (op.flags & CTTS_WE_TRIM) L = 0;   // trimming may shrink the region by any amount
                    if (op.flags & CTTS_WE_INTON) {
                        // the contour kernel stages CONTOUR_AHEAD samples past a tile: factors come from
                        // clamp_pitch(1 +- max_pitch_change) (ctts.c:2589), 0.9 .. 1.1 as shipped
                        const float lo = std::min(op.f0, std::min(op.f1, op.f2)), hi = std::max(op.f0, std::max(op.f1, op.f2));
                        if (!(lo >= 0.0f) || !(hi <= 2.05f)) sc->bad_factor = true;
                    }
                    break;
                case CTTS_OP_MARK:
                    close_region();
                    break;
                default:
                    return CTTS_GPU_ERR_INVALID_ARG;
            }
        }
        close_region();
        pre_out[u] = total;
        if (!std::isfinite(plan->speed[u])) return CTTS_GPU_ERR_INVALID_ARG;   // (size_t)(128 / NaN) is undefined in the reference too
        uint32_t hop = 0;
        const bool st = needs_stretch(plan->speed[u], &hop);
        sc->any_stretch |= st;
        bound_out[u] = st ? stretch_bound(total, hop) : total;
    }
    return 0;
}

// pass A, on a few host threads for large plans (it is serial work in front of the first launch)
int scan_plan(const ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, uint64_t big_threshold, PlanScan* sc, uint32_t* bad_utt) {
    const uint32_t n = plan->n_utts;
    sc->pre.assign(n, 0);
    sc->bound.assign(n, 0);
    uint32_t T = 1;
    if (plan->n_ops > (1u << 17)) {
        T = std::min<uint32_t>(4, std::max(1u, std::thread::hardware_concurrency()));
        if (ctx->knobs.host_threads) T = (uint32_t)ctx->knobs.host_threads;
    }
    if (T <= 1) return scan_range(ctx, plan, big_threshold, sc, bad_utt, 0, n, sc->pre.data(), sc->bound.data());
    std::vector<PlanScan> part(T);
    std::vector<int> rc(T, 0);
    std::vector<uint32_t> bad(T, 0);
    std::vector<std::thread> th;
    for (uint32_t t = 0; t < T; t++) {
        const uint32_t u0 = (uint32_t)((uint64_t)n * t / T), u1 = (uint32_t)((uint64_t)n * (t + 1) / T);
        th.emplace_back([&, t, u0, u1] {
            rc[t] = scan_range(ctx, plan, big_threshold, &part[t], &bad[t], u0, u1, sc->pre.data(), sc->bound.data());
        });
    }
    for (auto& x : th) x.join();
    for (uint32_t t = 0; t < T; t++) {
        if (rc[t]) {
            *bad_utt = bad[t];
            return rc[t];
        }
        sc->xf_max = std::max(sc->xf_max, part[t].xf_max);
        sc->region_max = std::max(sc->region_max, part[t].region_max);
        sc->big_region_max = std::max(sc->big_region_max, part[t].big_region_max);
        sc->n_regions += part[t].n_regions;
        sc->n_big_regions += part[t].n_big_regions;
        sc->bad_factor |= part[t].bad_factor;
        sc->any_stretch |= part[t].any_stretch;
    }
    return 0;
}

}  // namespace

extern "C" {

int ctts_gpu_init(ctts_gpu_ctx** out, const void* voice_db, size_t db_size, int device_ordinal) {
    if (!out || !voice_db || db_size < sizeof(DbHeader)) return fail(nullptr, CTTS_GPU_ERR_INVALID_ARG, "ctts_gpu_init: invalid argument");
    *out = nullptr;
    DbHeader h;
    memcpy(&h, voice_db, sizeof h);
    if (h.magic != 0x53545443u) return fail(nullptr, CTTS_GPU_ERR_INVALID_FORMAT, "ctts_gpu_init: not a voice.db (magic %08x)", h.magic);
    if (h.version != 1u) return fail(nullptr, CTTS_GPU_ERR_VERSION, "ctts_gpu_init: voice.db version %u", h.version);
    if ((uint64_t)h.index_offset + (uint64_t)h.unit_count * sizeof(DbEntry) > db_size ||
        (uint64_t)h.audio_offset + 2ull * h.total_samples > db_size)
        return fail(nullptr, CTTS_GPU_ERR_INVALID_FORMAT, "ctts_gpu_init: voice.db is truncated (%zu bytes)", db_size);

    int ndev = 0;
    {
        const cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev <= 0 || device_ordinal < 0 || device_ordinal >= ndev)   // no CPU fallback by design
            return fail(nullptr, CTTS_GPU_ERR_CUDA, "ctts_gpu_init: no CUDA device %d (%d visible%s%s): the back end has no CPU fallback",
                        device_ordinal, ndev, e != cudaSuccess ? ", " : "", e != cudaSuccess ? cudaGetErrorString(e) : "");
    }

    ctts_gpu_ctx* ctx = new ctts_gpu_ctx();
    ctx->device = device_ordinal;
    ctx->knobs.read_env();
    auto bail = [&](int code) {
        ctts_gpu_free(ctx);
        return code;
    };
#define CUI(call)                                                            \
    do {                                                                     \
        cudaError_t e_ = (call);                                             \
        if (e_ != cudaSuccess) {                                             \
            fail(nullptr, CTTS_GPU_ERR_CUDA, "ctts_gpu_init: %s: %s", #call, cudaGetErrorString(e_)); \
            return bail(CTTS_GPU_ERR_CUDA);                                  \
        }                                                                    \
    } while (0)
    CUI(cudaSetDevice(device_ordinal));
    CUI(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    CUI(cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device_ordinal));
    CUI(cudaDeviceGetAttribute(&ctx->smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device_ordinal));
    CUI(cudaDeviceGetAttribute(&ctx->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device_ordinal));
    // once per device: plans of different window sizes may be alive at the same time
    CUI(cudaFuncSetAttribute(ctts::assemble_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_optin));
    CUI(cudaFuncSetAttribute(ctts::wsola_verify_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ctts::WvSmem)));

    // re-pack: every unit starts on a 16-byte boundary, zero padded (int16x8 loads)
    const uint8_t* base = static_cast<const uint8_t*>(voice_db);
    const uint8_t* pcm = base + h.audio_offset;  // may be 2-byte misaligned (SURVEY.md 7.3)
    ctx->n_units = h.unit_count;
    ctx->unit_cnt.resize(h.unit_count);
    std::vector<uint32_t>& unit_off = ctx->unit_off;
    unit_off.resize(h.unit_count);
    uint64_t packed = 0;
    for (uint32_t u = 0; u < h.unit_count; u++) {
        DbEntry e;
        memcpy(&e, base + h.index_offset + (size_t)u * sizeof(DbEntry), sizeof e);
        if ((uint64_t)e.audio_offset + e.sample_count > h.total_samples) {
            fail(nullptr, CTTS_GPU_ERR_INVALID_FORMAT, "ctts_gpu_init: unit %u lies outside the PCM pool", u);
            return bail(CTTS_GPU_ERR_INVALID_FORMAT);
        }
        ctx->unit_cnt[u] = e.sample_count;
        unit_off[u] = (uint32_t)packed;
        packed += up8(e.sample_count);
        ctx->max_unit = std::max(ctx->max_unit, e.sample_count);
        if (packed > 0xffffffffull) {
            fail(nullptr, CTTS_GPU_ERR_INVALID_FORMAT, "ctts_gpu_init: more than 2^32 samples");
            return bail(CTTS_GPU_ERR_INVALID_FORMAT);
        }
    }
    std::vector<int16_t> pool(std::max<uint64_t>(packed, 8), 0);
    for (uint32_t u = 0; u < h.unit_count; u++) {
        DbEntry e;
        memcpy(&e, base + h.index_offset + (size_t)u * sizeof(DbEntry), sizeof e);
        memcpy(pool.data() + unit_off[u], pcm + 2ull * e.audio_offset, 2ull * e.sample_count);
    }
    ctx->pool_samples = pool.size();
    CUI(cudaMalloc(reinterpret_cast<void**>(&ctx->d_pool), pool.size() * sizeof(int16_t)));
    CUI(cudaMemcpy(ctx->d_pool, pool.data(), pool.size() * sizeof(int16_t), cudaMemcpyHostToDevice));
    CUI(cudaMalloc(reinterpret_cast<void**>(&ctx->d_unit_off), std::max<size_t>(h.unit_count, 1) * 4));
    CUI(cudaMalloc(reinterpret_cast<void**>(&ctx->d_unit_cnt), std::max<size_t>(h.unit_count, 1) * 4));
    if (h.unit_count) {
        CUI(cudaMemcpy(ctx->d_unit_off, unit_off.data(), h.unit_count * 4ull, cudaMemcpyHostToDevice));
        CUI(cudaMemcpy(ctx->d_unit_cnt, ctx->unit_cnt.data(), h.unit_count * 4ull, cudaMemcpyHostToDevice));
    }
    std::vector<float> tab(3 * 1024 + 256 + 512 + 4 * 1024);
    ctts_host_tables(tab.data(), tab.data() + 1024, tab.data() + 2048, tab.data() + 3072, tab.data() + 3328);
    for (int k = 0; k < 1024; k++) {   // interleaved crossfade table: one 16-byte load per sample
        const int k1 = k + 1 < 1024 ? k + 1 : 1023;
        float* e = tab.data() + 3840 + 4 * k;
        e[0] = tab[k];
        e[1] = tab[k1];
        e[2] = tab[1024 + k];
        e[3] = tab[1024 + k1];
    }
    CUI(cudaMalloc(reinterpret_cast<void**>(&ctx->d_tables), tab.size() * sizeof(float)));
    CUI(cudaMemcpy(ctx->d_tables, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice));
#undef CUI
    *out = ctx;
    return CTTS_GPU_OK;
}

void ctts_gpu_free(ctts_gpu_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->session) ctts_gpu_session_end(ctx->session, nullptr);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    cudaFree(ctx->d_pool);
    cudaFree(ctx->d_unit_off);
    cudaFree(ctx->d_unit_cnt);
    cudaFree(ctx->d_tables);
    for (ctts_gpu_ctx::RsTable* t : ctx->rs_tables) {
        cudaFree(t->d_taps);
        delete t;
    }
    for (ctts_gpu_ctx::LdTable* t : ctx->ld_tables) delete t;
    cudaFree(ctx->d_ld_gains);
    for (ctts_gpu_ctx::NormPool* np : ctx->norm_pools) {
        cudaFree(np->d_pool);
        cudaFree(np->d_meta);
        cudaFree(np->d_pitch);
        delete np;
    }
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    for (ctts_gpu_ctx::Lane& l : ctx->lane) {
        if (l.plan) ctts_gpu_plan_destroy(l.plan);
        cudaFree(l.arena.d);
        if (l.arena.h) cudaFreeHost(l.arena.h);
        cudaFree(l.d_out);
        cudaFree(l.d_rs);
        cudaFree(l.d_pack);
        cudaFree(l.d_pack_off);
        cudaFree(l.d_frames);
        cudaFree(l.d_flac_info);
        if (l.h_res) cudaFreeHost(l.h_res);
        if (l.kernels_done) cudaEventDestroy(l.kernels_done);
        if (l.counts_ready) cudaEventDestroy(l.counts_ready);
        if (l.copied) cudaEventDestroy(l.copied);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int ctts_gpu_set_stream(ctts_gpu_ctx* ctx, void* cuda_stream) {
    if (!ctx) return CTTS_GPU_ERR_INVALID_ARG;
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return CTTS_GPU_OK;
}

}  // extern "C"

namespace {

// The loudness setting (target, ceiling) at the context's current output rate: found among the context's tables or
// built.  The transitions A^len of the scan come from running the cascade itself on the unit states.
void ld_select(ctts_gpu_ctx* ctx, float target, float ceiling, bool true_peak) {
    const uint32_t hz = ctx->rs ? ctx->rs->hz : (uint32_t)CTTS_PLAN_SAMPLE_RATE;
    for (ctts_gpu_ctx::LdTable* t : ctx->ld_tables)
        if (t->hz == hz && t->target == target && t->ceiling == ceiling && t->true_peak == true_peak) {
            ctx->ld = t;
            return;
        }
    ctts_gpu_ctx::LdTable* t = new ctts_gpu_ctx::LdTable();
    t->hz = hz;
    t->target = target;
    t->ceiling = ceiling;
    t->true_peak = true_peak;
    t->ceiling_q = ctts_host_loudness_ceiling(ceiling);
    if (true_peak) {
        float h[49];
        ctts_host_true_peak_taps(h);
        for (int r = 1; r <= 3; r++)
            for (int i = 0; i < 12; i++) t->tp_h[r - 1][i] = h[44 - 4 * i + r];
    }
    double shelf[5], hp[2];
    ctts_host_loudness_filter(hz, shelf, hp);
    ctts::LdFilter& f = t->f;
    f.b0 = shelf[0] / 32768.0;
    f.b1 = shelf[1] / 32768.0;
    f.b2 = shelf[2] / 32768.0;
    f.a1 = shelf[3];
    f.a2 = shelf[4];
    f.h1 = hp[0];
    f.h2 = hp[1];
    f.fs = hz;
    f.lo = hz / 10;
    for (int r = 0; r < 2; r++)
        for (int i = 0; i < 4; i++) {
            double v[4] = {0.0, 0.0, 0.0, 0.0};
            v[i] = 1.0;
            ctts::LdState s{v[0], v[1], v[2], v[3]};
            for (uint32_t j = 0; j < f.lo + (uint32_t)r; j++) ctts::ld_step(f, s, 0.0);
            f.pw[r][0 * 4 + i] = s.s1;
            f.pw[r][1 * 4 + i] = s.s2;
            f.pw[r][2 * 4 + i] = s.t1;
            f.pw[r][3 * 4 + i] = s.t2;
        }
    ctx->ld_tables.push_back(t);
    ctx->ld = t;
}

// after a change of the output rate: the loudness setting moves to the new rate
int ld_follow_rate(ctts_gpu_ctx* ctx) {
    if (ctx->ld) ld_select(ctx, ctx->ld->target, ctx->ld->ceiling, ctx->ld->true_peak);
    return CTTS_GPU_OK;
}

}  // namespace

extern "C" {

int ctts_gpu_set_output_rate(ctts_gpu_ctx* ctx, uint32_t hz) {
    if (!ctx) return CTTS_GPU_ERR_INVALID_ARG;
    if (hz < 8000 || hz > 48000) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "output rate %u Hz outside [8000, 48000]", hz);
    const uint32_t g = std::gcd<uint32_t>(CTTS_PLAN_SAMPLE_RATE, hz), L = hz / g, M = CTTS_PLAN_SAMPLE_RATE / g, R = std::max(L, M);
    if (R > 1024) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "output rate %u Hz: the ratio %u/%u is not reduced enough (max(L, M) > 1024)", hz, L, M);
    if (ctx->session) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "the output rate cannot change while a session is open");
    if (hz == CTTS_PLAN_SAMPLE_RATE) {
        ctx->rs = nullptr;
        return ld_follow_rate(ctx);
    }
    for (ctts_gpu_ctx::RsTable* t : ctx->rs_tables)
        if (t->hz == hz) {
            ctx->rs = t;
            return ld_follow_rate(ctx);
        }
    CU(ctx, cudaSetDevice(ctx->device));
    const uint32_t N = 2u * 40u * R + 1u;
    std::vector<float> taps(N);
    ctts_host_resample_taps(L, M, taps.data());
    uint32_t kp, c, smem_floats, tiles;
    ctts_host_resample_geometry(L, M, 0, &kp, &c, &smem_floats, &tiles);
    // by phase, each row in the order the kernel walks it (resample.cuh), zero padded in front to a multiple of 4
    std::vector<float> rows((size_t)L * kp, 0.0f);
    for (uint32_t phi = 0; phi < L; phi++)
        for (uint32_t k = 0; k < kp; k++) {
            const uint64_t i = (uint64_t)phi + (uint64_t)L * (kp - 1 - k);
            if (i < N) rows[(size_t)phi * kp + k] = taps[i];
        }
    const int smem_bytes = (int)(smem_floats * sizeof(float));
    if (smem_bytes > ctx->smem_optin) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "output rate %u Hz: staging of %d bytes", hz, smem_bytes);
    if (smem_bytes > ctx->rs_smem_attr) {
        CU(ctx, cudaFuncSetAttribute(ctts::resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        ctx->rs_smem_attr = smem_bytes;
    }
    ctts_gpu_ctx::RsTable* t = new ctts_gpu_ctx::RsTable();
    t->hz = hz;
    t->L = L;
    t->M = M;
    t->kp = kp;
    t->c = c;
    t->smem_floats = smem_floats;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&t->d_taps), rows.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(t->d_taps, rows.data(), rows.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(t->d_taps);
        delete t;
        return fail(ctx, CTTS_GPU_ERR_CUDA, "output rate %u Hz: tap table: %s", hz, cudaGetErrorString(e));
    }
    ctx->rs_tables.push_back(t);
    ctx->rs = t;
    return ld_follow_rate(ctx);
}

// ctts_gpu_set_loudness and ctts_gpu_set_loudness_true_peak: the same rules, the ceiling kind apart
static int ld_set(ctts_gpu_ctx* ctx, float target_lufs, float ceiling_db, bool true_peak) {
    if (!ctx) return CTTS_GPU_ERR_INVALID_ARG;
    if (!std::isfinite(target_lufs) || (target_lufs != 0.0f && (target_lufs < -60.0f || target_lufs > -5.0f)))
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "loudness target %g LUFS: neither 0 nor in [-60, -5]", (double)target_lufs);
    if (!std::isfinite(ceiling_db) || ceiling_db < -20.0f || ceiling_db > 0.0f)
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "peak ceiling %g %s outside [-20, 0]", (double)ceiling_db, true_peak ? "dBTP" : "dBFS");
    if (ctx->session) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "the loudness setting cannot change while a session is open");
    if (target_lufs == 0.0f) {
        ctx->ld = nullptr;
        return CTTS_GPU_OK;
    }
    if (!ctx->d_ld_gains) {
        std::vector<uint32_t> gains(2 * ctts::LD_K_MAX + 1);
        ctts_host_loudness_gains(gains.data());
        CU(ctx, cudaSetDevice(ctx->device));
        cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ctx->d_ld_gains), gains.size() * 4);
        if (e == cudaSuccess) e = cudaMemcpy(ctx->d_ld_gains, gains.data(), gains.size() * 4, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            cudaFree(ctx->d_ld_gains);
            ctx->d_ld_gains = nullptr;
            return fail(ctx, CTTS_GPU_ERR_CUDA, "loudness gain table: %s", cudaGetErrorString(e));
        }
    }
    ld_select(ctx, target_lufs, ceiling_db, true_peak);
    return CTTS_GPU_OK;
}

int ctts_gpu_set_loudness(ctts_gpu_ctx* ctx, float target_lufs, float ceiling_dbfs) {
    return ld_set(ctx, target_lufs, ceiling_dbfs, false);
}

int ctts_gpu_set_loudness_true_peak(ctts_gpu_ctx* ctx, float target_lufs, float ceiling_dbtp) {
    return ld_set(ctx, target_lufs, ceiling_dbtp, true);
}

const char* ctts_gpu_last_error(const ctts_gpu_ctx* ctx) { return ctx ? ctx->err : g_init_err; }

void* ctts_gpu_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) return nullptr;
    return p;
}

void ctts_gpu_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

int ctts_gpu_plan_bounds(const ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, uint64_t* out_bound) {
    if (!ctx || !plan || !out_bound) return CTTS_GPU_ERR_INVALID_ARG;
    if (plan->n_utts && (!plan->utt_op_begin || !plan->speed)) return CTTS_GPU_ERR_INVALID_ARG;
    PlanScan sc;
    uint32_t bad = 0;
    int rc = scan_plan(ctx, plan, ~0ull, &sc, &bad);
    if (rc) return rc;
    for (uint32_t u = 0; u < plan->n_utts; u++) out_bound[u] = rate_bound(ctx->rs, sc.bound[u]);
    return CTTS_GPU_OK;
}

void ctts_gpu_plan_destroy(ctts_gpu_plan* p) {
    if (!p) return;
    if (p->ctx && (!p->arena || !p->owned.empty())) {
        // (a piece of a session is destroyed after its lane's events: nothing of it is still running)
        cudaSetDevice(p->ctx->device);
        cudaStreamSynchronize(p->ctx->stream);
    }
    if (p->d_prof) {
        unsigned long long h[16];
        if (cudaMemcpy(h, p->d_prof, sizeof h, cudaMemcpyDeviceToHost) == cudaSuccess) {
            static const char* const names[5] = {"canonical region", "copied whole", "resumed at the contour", "assembled in the window", "assembled in HBM"};
            unsigned long long tot = 0;
            for (int i = 0; i < 5; i++) tot += h[2 * i];
            fprintf(stderr, "ctts_gpu: CTA time per task class, all launches of this plan (%.1f ms of CTA time)\n", tot * 1e-6);
            for (int i = 0; i < 5; i++)
                if (h[2 * i + 1])
                    fprintf(stderr, "  %-26s %9llu tasks  %6.2f %% of the time  %7.2f us per task\n", names[i], h[2 * i + 1],
                            100.0 * h[2 * i] / (tot ? tot : 1), h[2 * i] * 1e-3 / h[2 * i + 1]);
            if (h[11]) fprintf(stderr, "  (WORD_END ops inside HBM tasks: %llu, %.2f us each, %.2f %% of the time)\n", h[11], h[10] * 1e-3 / h[11], 100.0 * h[10] / (tot ? tot : 1));
        }
    }
    for (void* d : p->owned) cudaFree(d);
    cudaFree(p->d_out_owned);
    cudaFree(p->d_nat_owned);
    delete p;
}

}  // extern "C"

namespace {

// Workspace of one plan.  Device buffers: individual cudaMallocs (resident plans), or bump allocation from
// a lane's grow-only arena (session pieces: no malloc/free per call).  Upload staging: bump allocation from
// the arena's pinned block, or from the plan's pageable h_staging.  A measuring PlanAlloc allocates nothing
// and returns nullptr: it only counts the bytes, so that one list of buffers both sizes and lays out the workspace.
struct PlanAlloc {
    ctts_gpu_plan* p;
    bool measure;
    size_t d_used = 0, staged = 0;   // bytes
    cudaError_t err = cudaSuccess;   // cudaErrorMemoryAllocation also when the list outgrows the arena

    static size_t up256(size_t v) { return (v + 255) & ~(size_t)255; }

    template <typename T>
    T* host(size_t count) {
        const size_t bytes = up256(std::max<size_t>(count, 1) * sizeof(T));
        staged += bytes;
        if (measure) return nullptr;
        char* const base = p->arena ? p->arena->h : p->h_staging.data();
        if (staged > (p->arena ? p->arena->h_cap : p->h_staging.size())) { err = cudaErrorMemoryAllocation; return nullptr; }
        return reinterpret_cast<T*>(base + staged - bytes);
    }

    template <typename T>
    T* dev(size_t count) {
        const size_t bytes = up256(std::max<size_t>(count, 1) * sizeof(T));
        if (measure || p->arena) {
            d_used += bytes;
            if (measure) return nullptr;
            if (d_used > p->arena->d_cap) { err = cudaErrorMemoryAllocation; return nullptr; }
            return reinterpret_cast<T*>(p->arena->d + d_used - bytes);
        }
        void* d = nullptr;
        cudaError_t e = cudaMalloc(&d, bytes);
        if (e != cudaSuccess) { err = e; return nullptr; }
        p->owned.push_back(d);
        return static_cast<T*>(d);
    }
};

int ensure_arena(ctts_gpu_ctx* ctx, Arena* a, size_t d_bytes, size_t h_bytes) {
    if (d_bytes > a->d_cap) {
        cudaFree(a->d);
        a->d = nullptr;
        a->d_cap = 0;
        const size_t cap = d_bytes + d_bytes / 4;
        if (cudaMalloc(reinterpret_cast<void**>(&a->d), cap) != cudaSuccess)
            return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "device workspace of %zu bytes", cap);
        a->d_cap = cap;
    }
    if (h_bytes > a->h_cap) {
        if (a->h) cudaFreeHost(a->h);
        a->h = nullptr;
        a->h_cap = 0;
        const size_t cap = h_bytes + h_bytes / 4;
        if (cudaHostAlloc(reinterpret_cast<void**>(&a->h), cap, cudaHostAllocDefault) != cudaSuccess)
            return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "pinned staging of %zu bytes", cap);
        a->h_cap = cap;
    }
    return 0;
}

#define CUP(call)                                                                               \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            ctts_gpu_plan_destroy(p);                                                           \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? CTTS_GPU_ERR_OUT_OF_MEMORY : CTTS_GPU_ERR_CUDA, \
                        "%s: %s", #call, cudaGetErrorString(e_));                               \
        }                                                                                       \
    } while (0)

// The normalized pool for `target_rms` (bit pattern compared: the kernel's result depends on nothing
// else), created on the context stream at first use.
int norm_pool_for(ctts_gpu_ctx* ctx, float target_rms, ctts_gpu_ctx::NormPool** out) {
    for (ctts_gpu_ctx::NormPool* np : ctx->norm_pools)
        if (memcmp(&np->target_rms, &target_rms, sizeof(float)) == 0) {
            *out = np;
            return CTTS_GPU_OK;
        }
    if (ctx->norm_pools.size() >= 64)
        return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "more than 64 distinct target_rms values in one context");
    ctts_gpu_ctx::NormPool* np = new ctts_gpu_ctx::NormPool();
    np->target_rms = target_rms;
    np->pitch_cap = std::max<uint32_t>(1u << 16, 64u * ctx->n_units);
    if (ctx->knobs.pitch_slots) np->pitch_cap = (uint32_t)ctx->knobs.pitch_slots;
    np->pitch_slots.resize(ctx->n_units);
    if (cudaMalloc(reinterpret_cast<void**>(&np->d_pool), std::max<uint64_t>(ctx->pool_samples, 8) * sizeof(int16_t)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&np->d_meta), std::max<size_t>(ctx->n_units, 1) * sizeof(int4)) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void**>(&np->d_pitch), (size_t)np->pitch_cap * sizeof(float)) != cudaSuccess) {
        cudaFree(np->d_pool);
        cudaFree(np->d_meta);
        cudaFree(np->d_pitch);
        delete np;
        return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "normalized pool");
    }
    const auto t0 = std::chrono::steady_clock::now();
    cudaError_t ce = cudaMemsetAsync(np->d_pitch, 0, (size_t)np->pitch_cap * sizeof(float), ctx->stream);
    if (ce == cudaSuccess && ctx->n_units) {
        ctts::normalize_pool_kernel<<<ctx->n_units, ctts::ASM_THREADS, 0, ctx->stream>>>(ctx->d_pool, np->d_pool, ctx->d_unit_off,
                                                                                       ctx->d_unit_cnt, np->d_meta, target_rms);
        ce = cudaGetLastError();
    }
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);   // once: later plans may run on another stream
    if (ce != cudaSuccess) {   // the pool is registered only once it is filled
        cudaFree(np->d_pool);
        cudaFree(np->d_meta);
        cudaFree(np->d_pitch);
        delete np;
        return fail(ctx, CTTS_GPU_ERR_CUDA, "normalize_pool_kernel: %s", cudaGetErrorString(ce));
    }
    ctx->norm_pools.push_back(np);
    if (ctx->knobs.trace)
        fprintf(stderr, "ctts_gpu: normalized pool for target_rms %g: %u units, %llu samples in %.2f ms\n", (double)target_rms, ctx->n_units,
                (unsigned long long)ctx->pool_samples, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    *out = np;
    return CTTS_GPU_OK;
}

// Table slot (+1) of the pitch of unit u's head over R samples; a new pair is appended to `jobs`
// for unit_pitch_kernel.  0: the table is full (the kernel then estimates the head itself).
inline uint32_t pitch_slot_for(ctts_gpu_ctx* ctx, ctts_gpu_ctx::NormPool* np, uint32_t u, uint32_t R, std::vector<uint3>* jobs) {
    std::vector<std::pair<uint32_t, uint32_t>>& v = np->pitch_slots[u];
    for (const std::pair<uint32_t, uint32_t>& e : v)
        if (e.first == R) return e.second + 1;
    if (np->pitch_used >= np->pitch_cap) return 0;
    const uint32_t slot = np->pitch_used++;
    v.emplace_back(R, slot);
    jobs->push_back(make_uint3(ctx->unit_off[u], R, slot));
    return slot + 1;
}

// Fill the table slots of `jobs` (rare: only for pairs no earlier plan of this context used).
int run_pitch_jobs(ctts_gpu_ctx* ctx, ctts_gpu_ctx::NormPool* np, const std::vector<uint3>& jobs) {
    if (jobs.empty()) return CTTS_GPU_OK;
    const auto t0 = std::chrono::steady_clock::now();
    uint3* d_jobs = nullptr;
    CU(ctx, cudaMalloc(reinterpret_cast<void**>(&d_jobs), jobs.size() * sizeof(uint3)));
    cudaError_t e = cudaMemcpyAsync(d_jobs, jobs.data(), jobs.size() * sizeof(uint3), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) {
        ctts::unit_pitch_kernel<<<(unsigned)jobs.size(), ctts::ASM_THREADS, 0, ctx->stream>>>(np->d_pool, d_jobs, np->d_pitch);
        e = cudaGetLastError();
    }
    // the slots are used by every later launch, on whichever stream: finish them now
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_jobs);
    if (e != cudaSuccess) return fail(ctx, CTTS_GPU_ERR_CUDA, "unit_pitch_kernel: %s", cudaGetErrorString(e));
    if (ctx->knobs.trace)
        fprintf(stderr, "ctts_gpu: unit-head pitch table: %zu new entries (%u in all) in %.2f ms including the stream drain\n", jobs.size(),
                np->pitch_used, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    return CTTS_GPU_OK;
}

// Slots packed by their bounds, up8(bound) + 8 samples each: the n + 1 offsets.
int pack_slots(ctts_gpu_ctx* ctx, const std::vector<uint64_t>& bound, std::vector<uint64_t>* off) {
    off->resize(bound.size() + 1);
    uint64_t o = 0;
    for (uint32_t u = 0; u < bound.size(); u++) {
        if (bound[u] + 16 > 0xffffffffull)
            return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "utterance %u too long (%llu samples)", u, (unsigned long long)bound[u]);
        (*off)[u] = o;
        o += up8(bound[u]) + 8;
    }
    off->back() = o;
    return CTTS_GPU_OK;
}

// The plan compiler, part 1: validation, bounds, output layout, workspace.  One launch of every kernel
// per plan; a large batch is cut into pieces (plans) by the session code below.  `arena` != nullptr:
// device / pinned workspace comes from that lane's grow-only arena.  build_tasks() is part 2.
int prepare_plan(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, const ctts_assembly_params* params,
                 const uint64_t* out_offsets, Arena* arena, ctts_gpu_plan** out) {
    if (!ctx || !plan || !params || !out) return CTTS_GPU_ERR_INVALID_ARG;
    if (plan->n_utts && (!plan->utt_op_begin || !plan->speed)) return CTTS_GPU_ERR_INVALID_ARG;
    if (plan->n_ops && !plan->ops) return CTTS_GPU_ERR_INVALID_ARG;
    if (params->min_silence_samples < 10)
        // below 10 the reference's keep = max(min/4, 10) overruns the silent run (SURVEY.md app. A)
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "min_silence_samples < 10 is not memory-safe in the reference");
    *out = nullptr;
    CU(ctx, cudaSetDevice(ctx->device));
    const uint32_t n = plan->n_utts;

    // ---- pass A
    const uint64_t scr_samples = (uint64_t)(ctts::SCR_WORDS - 4) / 2 * 32;   // region length the shared trim mask covers
    PlanScan sc;
    uint32_t bad = 0;
    int rc = scan_plan(ctx, plan, scr_samples, &sc, &bad);
    if (rc) return fail(ctx, rc, "invalid plan (utterance %u)", bad);
    if (sc.bad_factor) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "WORD_END pitch factors must lie in [0, 2.05]");
    const std::vector<uint64_t>& pre = sc.pre;
    ctts_gpu_ctx::RsTable* const rs = ctx->rs;
    std::vector<uint64_t> bound(sc.bound);   // at the output rate
    if (rs)
        for (uint64_t& b : bound) b = rate_bound(rs, b);

    ctts_gpu_ctx::NormPool* np = nullptr;
    rc = norm_pool_for(ctx, params->target_rms, &np);
    if (rc) return rc;

    ctts_gpu_plan* p = new ctts_gpu_plan();
    p->ctx = ctx;
    p->np = np;
    p->n_utts = n;
    p->prm = *params;
    p->bounds = bound;
    p->rs = rs;
    p->arena = arena;
    p->op0 = n ? plan->utt_op_begin[0] : 0;
    const uint32_t n_ops_local = n ? plan->utt_op_begin[n] - p->op0 : 0;   // (validated by the scan)

    // ---- output layout
    if (out_offsets) {
        p->offsets.assign(out_offsets, out_offsets + (size_t)n + 1);
        for (uint32_t u = 0; u < n; u++) {
            if ((out_offsets[u] & 7) || out_offsets[u + 1] < out_offsets[u] ||
                out_offsets[u + 1] - out_offsets[u] < bound[u] || out_offsets[u + 1] - out_offsets[u] > 0xffffffffull) {
                delete p;
                return fail(ctx, CTTS_GPU_ERR_BOUNDS, "output slot %u is misaligned or smaller than its bound %llu", u,
                            (unsigned long long)bound[u]);
            }
        }
    } else if ((rc = pack_slots(ctx, bound, &p->offsets)) != 0) {
        delete p;
        return rc;
    }
    if (rs) {
        // native slots packed by the native bounds; resample_kernel turns them into the slots above
        if ((rc = pack_slots(ctx, sc.bound, &p->n_offsets)) != 0) {
            delete p;
            return rc;
        }
        const uint64_t ob_max = n ? *std::max_element(bound.begin(), bound.end()) : 0;
        uint32_t kp, c, smem_floats;
        ctts_host_resample_geometry(rs->L, rs->M, ob_max, &kp, &c, &smem_floats, &p->rs_tiles);
    } else {
        p->n_offsets = p->offsets;
    }
    // loudness: one chunk per 100 ms sub-block that can start before the bound
    const ctts_gpu_ctx::LdTable* const ld = ctx->ld;
    p->ld = ld;
    // (true peak: and one ld_true_peak_kernel tile per LD_TP_TILE positions -6 .. bound + 5)
    std::vector<uint64_t> ld_chunk0, ld_tile0;
    const bool tp = ld && ld->true_peak;
    if (ld) {
        ld_chunk0.resize((size_t)n + 1, 0);
        uint64_t max_chunks = 0, max_bound = 0;
        for (uint32_t u = 0; u < n; u++) {
            const uint64_t k = (bound[u] * 10 + ld->hz - 1) / ld->hz;
            ld_chunk0[u + 1] = ld_chunk0[u] + k;
            max_chunks = std::max(max_chunks, k);
            max_bound = std::max(max_bound, bound[u]);
        }
        p->ld_tiles = (uint32_t)std::max<uint64_t>((max_chunks + ctts::LD_THREADS - 1) / ctts::LD_THREADS, 1);
        p->ld_apply_tiles = (uint32_t)std::max<uint64_t>((max_bound + ctts::LD_APPLY_TILE - 1) / ctts::LD_APPLY_TILE, 1);
        if (tp) {
            ld_tile0.resize((size_t)n + 1, 0);
            for (uint32_t u = 0; u < n; u++) ld_tile0[u + 1] = ld_tile0[u] + ctts::ld_tp_tiles(bound[u]);
            p->ld_tp_tiles = (uint32_t)ctts::ld_tp_tiles(max_bound);
        }
    }

    // ---- shared-memory geometry
    const uint32_t max_unit = ctx->max_unit, xf_max = sc.xf_max;
    const uint32_t hcap = (uint32_t)up8(std::max<uint32_t>(std::min(xf_max, max_unit), 496)) + 8;
    if (hcap > 2 * ctts::SCR_WORDS) {
        delete p;
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "crossfade of %u samples exceeds the staging capacity", xf_max);
    }
    auto smem_for = [&](uint32_t wcap) { return ctts::SMEM_HSTAGE + hcap * 2 + (wcap + 16) * 2; };
    // window: as large as the target occupancy allows, no larger than the largest region needs
    const int want_ctas = ctx->knobs.ctas_per_sm;
    const uint32_t budget = std::min<uint32_t>((uint32_t)ctx->smem_optin, (uint32_t)(ctx->smem_per_sm / want_ctas - 1024));
    uint32_t wcap = (uint32_t)up8(std::min<uint64_t>(sc.region_max + 16, 1u << 20));
    if (ctx->knobs.window) wcap = (uint32_t)up8(std::max(256, ctx->knobs.window));   // tests: force the HBM path
    while (wcap > 1024 && smem_for(wcap) > budget) wcap -= 256;
    wcap &= ~7u;
    if (smem_for(wcap) > (uint32_t)ctx->smem_optin) {
        delete p;
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "crossfade / unit sizes (%u, %u samples) do not fit shared memory", xf_max, max_unit);
    }
    p->wcap = wcap;
    p->hcap = hcap;
    p->smem_bytes = smem_for(wcap);

    // ---- slots of stretched utterances and WSOLA tasks, longest first
    std::vector<uint32_t> order;
    if (sc.any_stretch)
        for (uint32_t u = 0; u < n; u++) {
            uint32_t hop = 0;
            if (needs_stretch(plan->speed[u], &hop)) order.push_back(u);
        }
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return pre[a] > pre[b]; });
    std::vector<ctts::StretchTask> stasks;
    std::vector<uint32_t> ola_task, ola_first;
    p->pre_off.assign(n, ~0ull);
    p->pre_cap.assign(n, 0);
    uint64_t pre_total = 0, pos_total = 0;
    for (const uint32_t u : order) {
        uint32_t hop = 0;
        needs_stretch(plan->speed[u], &hop);
        if (pre[u] + 16 > 0xffffffffull) {
            delete p;
            return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "utterance %u too long", u);
        }
        p->pre_off[u] = pre_total;
        p->pre_cap[u] = (uint32_t)(up8(pre[u]) + 8);
        ctts::StretchTask st;
        st.utt = u;
        st.hop = hop;
        st.pre_off = pre_total;
        st.out_off = p->n_offsets[u];
        st.out_cap = (uint32_t)(p->n_offsets[u + 1] - p->n_offsets[u]);
        st.pos_off = (uint32_t)pos_total;
        st.max_frames = (uint32_t)(pre[u] > 512 ? (pre[u] - 512) / 128 + 1 : 1);
        if (st.max_frames > 1)
            p->verify_tiles = std::max(p->verify_tiles, (st.max_frames - 1 + ctts::WV_FRAMES - 1) / ctts::WV_FRAMES);
        const uint64_t used_max = (uint64_t)st.max_frames * hop + 512;
        const uint32_t per_block = ctts::ola_block_span(hop);
        for (uint64_t f = 0; f < used_max; f += per_block) {
            ola_task.push_back((uint32_t)stasks.size());
            ola_first.push_back((uint32_t)f);
        }
        stasks.push_back(st);
        pre_total += p->pre_cap[u];
        pos_total += st.max_frames;
        if (pos_total > 0xffffffffull) {
            delete p;
            return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "too many WSOLA frames in one batch");
        }
    }
    p->n_stretch = (uint32_t)stasks.size();
    p->n_ola_blocks = (uint32_t)ola_task.size();
    if (sc.n_regions + 1 > 0x7fffffffull) {
        delete p;
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "too many region tasks");
    }

    // ---- workspace: one list of device buffers and upload staging, run once to measure it (the arena, or the
    // pageable staging, is sized from that) and once to lay it out.  The private op copy and the tasks are built
    // directly in the staging.
    // merging only lowers the count of region tasks; canonical word regions (each stands for >= 2 tasks) add at most half
    const size_t tasks_cap = (size_t)sc.n_regions + (size_t)sc.n_regions / 2 + 2;
    ctts::StretchTask* h_st = nullptr;
    uint32_t *h_ot = nullptr, *h_of = nullptr;
    unsigned long long* h_off = nullptr;
    const size_t off_words = ((rs ? 2 : 1) + (ld ? 1 : 0) + (tp ? 1 : 0)) * ((size_t)n + 1);   // of d_off
    auto layout = [&](PlanAlloc& al) {
        p->d_ops = al.dev<ctts_plan_op>(n_ops_local);
        p->d_tasks = al.dev<ctts::RegionTask>(tasks_cap);
        p->d_chain = al.dev<unsigned long long>(tasks_cap);
        p->d_ticket = al.dev<uint32_t>(1);
        if (ctx->knobs.task_times && !arena) p->d_prof = al.dev<unsigned long long>(16);
        p->d_counts = al.dev<uint32_t>(n);
        p->d_pre_counts = al.dev<uint32_t>(n);
        p->d_err = al.dev<uint32_t>(n);
        p->d_off = al.dev<unsigned long long>(off_words);
        p->d_final_counts = p->d_counts;
        if (rs) {
            p->d_rs_counts = al.dev<uint32_t>(n);
            p->d_final_counts = p->d_rs_counts;
        }
        if (ld) {
            const uint64_t chunks = ld_chunk0[n];
            p->d_ld_state = al.dev<double>(4 * chunks);
            p->d_ld_energy = al.dev<double>(chunks);
            p->d_ld_peak = al.dev<uint32_t>(chunks);
            p->d_ld_lufs = al.dev<double>(n);
            p->d_ld_gain = al.dev<uint32_t>(n);
            if (tp) {
                p->d_ld_tp_tile = al.dev<float>(ld_tile0[n]);
                p->d_ld_tp = al.dev<float>(n);
            }
        }
        if (p->n_stretch) {
            p->d_stasks = al.dev<ctts::StretchTask>(stasks.size());
            p->d_ola_task = al.dev<uint32_t>(ola_task.size());
            p->d_ola_first = al.dev<uint32_t>(ola_first.size());
            p->d_pre = al.dev<int16_t>(pre_total);
            p->d_frame_pos = al.dev<uint32_t>(pos_total);
            p->d_n_frames = al.dev<uint32_t>(5 * (size_t)p->n_stretch);   // frames, exact evaluations, first bad frame, first silent frame, tier-2 candidates
        }
        p->h_ops = al.host<ctts_plan_op>(n_ops_local);
        p->h_tasks = al.host<ctts::RegionTask>(tasks_cap);
        if (p->n_stretch) {
            h_st = al.host<ctts::StretchTask>(stasks.size());
            h_ot = al.host<uint32_t>(ola_task.size());
            h_of = al.host<uint32_t>(ola_first.size());
        }
        h_off = al.host<unsigned long long>(off_words);
    };
    PlanAlloc al{p, true};
    layout(al);
    if (arena) {
        // + the region store, carved by build_tasks once the regions are known; reserved here at its upper bound:
        // the canonical regions' slots and the shared whole tasks' + their tables.  A slot takes up8(bound) + 8
        // samples and every slot can be charged to a task of its own: a canonical region (a group of >= 2 tasks) to
        // the task whose bound sizes it, a shared whole task (>= 2 tasks with equal ops, so equal bounds) to one of
        // its tasks that is not that first task of the group.  So the slots hold at most the sum of the bounds +
        // 16 samples per task, whatever the window (build_tasks still checks that the store fits the arena).
        const uint64_t pre_sum = std::accumulate(pre.begin(), pre.end(), (uint64_t)0);
        const size_t region_bytes = !ctx->knobs.region_dedup ? 0 :
            PlanAlloc::up256((pre_sum + 16 * (sc.n_regions + 2)) * sizeof(int16_t)) + 2 * PlanAlloc::up256((sc.n_regions + 2) * 8);
        rc = ensure_arena(ctx, arena, al.d_used + region_bytes, al.staged);
        if (rc) { delete p; return rc; }
    } else {
        p->h_staging.resize(al.staged);
    }
    al = PlanAlloc{p, false};
    layout(al);
    if (p->d_prof) cudaMemset(p->d_prof, 0, 16 * 8);
    if (sc.n_big_regions) {
        // rare (regions longer than ~51 k samples): always a separate allocation
        p->trim_words = (uint32_t)(2 * ((sc.big_region_max + 31) / 32) + 8);
        p->big_cap = (uint32_t)sc.n_big_regions;
        void* d = nullptr;
        if (cudaMalloc(&d, (size_t)p->big_cap * p->trim_words * 4) != cudaSuccess) al.err = cudaErrorMemoryAllocation;
        else { p->owned.push_back(d); p->d_trim = static_cast<uint32_t*>(d); }
    }
    if (al.err != cudaSuccess) {
        ctts_gpu_plan_destroy(p);
        return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "plan workspace: %s", cudaGetErrorString(al.err));
    }
    p->d_used = al.d_used;
    // arena: through the lane's pinned staging, truly asynchronous, no stream drain per piece (the staging is
    // reused only after the lane's piece has completed)
    cudaStream_t st = ctx->stream;
    CUP(cudaMemsetAsync(p->d_chain, 0, tasks_cap * 8, st));
    if (p->n_stretch) {
        memcpy(h_st, stasks.data(), stasks.size() * sizeof(ctts::StretchTask));
        memcpy(h_ot, ola_task.data(), ola_task.size() * 4);
        memcpy(h_of, ola_first.data(), ola_first.size() * 4);
        CUP(cudaMemcpyAsync(p->d_stasks, h_st, stasks.size() * sizeof(ctts::StretchTask), cudaMemcpyHostToDevice, st));
        CUP(cudaMemcpyAsync(p->d_ola_task, h_ot, ola_task.size() * 4, cudaMemcpyHostToDevice, st));
        CUP(cudaMemcpyAsync(p->d_ola_first, h_of, ola_first.size() * 4, cudaMemcpyHostToDevice, st));
    }
    unsigned long long* o = h_off;
    if (rs) o = std::copy(p->n_offsets.begin(), p->n_offsets.end(), o);
    o = std::copy(p->offsets.begin(), p->offsets.end(), o);
    if (ld) o = std::copy(ld_chunk0.begin(), ld_chunk0.end(), o);
    if (tp) std::copy(ld_tile0.begin(), ld_tile0.end(), o);
    CUP(cudaMemcpyAsync(p->d_off, h_off, off_words * 8, cudaMemcpyHostToDevice, st));
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ctts::assemble_kernel, ctts::ASM_THREADS, p->smem_bytes) != cudaSuccess || occ < 1)
        occ = 1;
    p->occ = (uint32_t)occ;

    p->info.n_stretch = p->n_stretch;
    p->info.bound_samples = std::accumulate(bound.begin(), bound.end(), (uint64_t)0);
    p->info.smem_bytes = p->smem_bytes;
    p->info.window_samples = wcap;
    p->info.halo_samples = hcap;
    p->info.threads = ctts::ASM_THREADS;
    p->info.ctas_per_sm = p->occ;
    *out = p;
    return CTTS_GPU_OK;
}

// The plan compiler, part 2: private op copy (with provably dead fade-outs turned into
// no-ops), regions -> tasks, ticket order, upload.  `plan` is the one prepare_plan() was given.
int build_tasks(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, const ctts_batch_plan* plan, cudaStream_t st) {
    const uint32_t n = p->n_utts;
    const uint32_t* ub = plan->utt_op_begin;
    const std::vector<uint32_t>& ucnt = ctx->unit_cnt;
    const uint32_t wcap = p->wcap;
    const uint64_t scr_samples = (uint64_t)(ctts::SCR_WORDS - 4) / 2 * 32;
    ctts_plan_op* h_ops = p->h_ops;
    const uint32_t op0 = p->op0;   // h_ops / d_ops hold the caller's ops from op0 on
    const uint32_t n_ops = n ? ub[n] - op0 : 0;
    if (n_ops) memcpy(h_ops, plan->ops + op0, (size_t)n_ops * sizeof(ctts_plan_op));

    // A fade-out that provably acts on zeros (or on an empty buffer) becomes a no-op, so that a
    // pause-only region never has to reach back into its predecessor's samples.  Trailing zeros:
    // appended silence stays zero under apply_fade_out (0 * g == 0); a unit, or a WORD_END over a
    // region that holds audio (trimming / the contour may move samples into the tail), resets it.
    // A region with no unit (a pause) or a tiny one is appended to the task before it while the
    // sum still fits the window.
    // base_lb: a LOWER bound of the utterance's sample count when the task starts (trimming may take a whole region
    // away, pauses and untrimmed regions stay): a task whose threshold it meets need not wait for its predecessor
    // before it starts
    struct HostTask { uint32_t op_begin, op_end; uint64_t bound; uint32_t region_max; uint64_t base_lb; };
    std::vector<HostTask> ht;
    std::vector<uint3> pitch_jobs;
    std::vector<uint32_t> pitch_job_units;   // unit of every new table entry (to take them back if the fill fails)
    std::vector<uint32_t> ht_begin(n + 1, 0);   // CSR: tasks of utterance u
    uint32_t max_rows = 0;
    for (uint32_t u = 0; u < n; u++) {
        ht_begin[u] = (uint32_t)ht.size();
        uint64_t tz = 0, count_ub = 0, rb = 0, L = 0;
        uint64_t count_lb = 0, word_lb = 0, region_lb = 0;   // lower bounds: of the count, at the last MARK, at the start of the open region
        uint32_t r_units = 0, r_begin = ub[u];
        bool audio = false;
        auto close_region = [&](uint32_t r_end) {
            if (r_end == r_begin) return;
            const bool tiny = r_units == 0 || rb <= 2048;
            if (ht.size() > ht_begin[u] && tiny && ht.back().bound + rb <= wcap) {
                ht.back().op_end = r_end;
                ht.back().bound += rb;
                ht.back().region_max = (uint32_t)std::max<uint64_t>(ht.back().region_max, rb);
            } else {
                ht.push_back(HostTask{r_begin, r_end, rb, (uint32_t)std::min<uint64_t>(rb, 0xffffffffull), region_lb});
            }
            region_lb = count_lb;
            r_begin = r_end;
            rb = 0;
            r_units = 0;
            L = 0;
        };
        for (uint32_t k = ub[u]; k < ub[u + 1]; k++) {
            ctts_plan_op& op = h_ops[k - op0];
            switch (op.kind) {
                case CTTS_OP_UNIT: {
                    const uint32_t cn = ucnt[op.a];
                    // private copy: the unit's length and pool offset ride in the (unused) float fields,
                    // so the kernel needs no dependent table look-up before the gather
                    memcpy(&op.f0, &cn, 4);
                    memcpy(&op.f1, &ctx->unit_off[op.a], 4);
                    // ... and so does the table slot of the head's pitch over min(2*xf, n/2) samples
                    // (the analysis length of ctts.c:1983-1987 whenever the buffer is long enough)
                    uint32_t slot1 = 0;
                    if (!(op.flags & CTTS_UNIT_AFTER_BOUNDARY) && op.b > 0 && cn >= 200) {
                        const uint32_t m2 = 2 * op.b < cn / 2 ? 2 * op.b : cn / 2;   // uint32 like the kernel
                        if (m2 >= 200) {
                            const size_t before = pitch_jobs.size();
                            slot1 = pitch_slot_for(ctx, p->np, op.a, m2, &pitch_jobs);
                            if (pitch_jobs.size() != before) pitch_job_units.push_back(op.a);
                        }
                    }
                    memcpy(&op.f2, &slot1, 4);
                    count_ub += cn;
                    count_lb += (op.flags & CTTS_UNIT_AFTER_BOUNDARY) ? cn : cn - std::min(op.b, cn);
                    p->info.gather_samples += cn;
                    rb += unit_append_bound(op, cn, L);
                    r_units++;
                    if (cn) { tz = 0; audio = true; }
                    break;
                }
                case CTTS_OP_SILENCE:
                    tz += op.a;
                    count_ub += op.a;
                    count_lb += op.a;
                    rb += op.a;
                    L += op.a;
                    break;
                case CTTS_OP_FADE_OUT:
                    if (count_ub == 0 || tz >= op.a) op.kind = ctts::OP_NOP;
                    break;
                case CTTS_OP_WORD_END:
                    if (audio) tz = 0;
                    if (op.flags & CTTS_WE_TRIM) { L = 0; count_lb = word_lb; }
                    break;
                case CTTS_OP_MARK:
                    audio = false;
                    word_lb = count_lb;
                    close_region(k + 1);
                    break;
            }
        }
        close_region(ub[u + 1]);
        max_rows = std::max<uint32_t>(max_rows, (uint32_t)ht.size() - ht_begin[u]);
    }
    ht_begin[n] = (uint32_t)ht.size();
    {
        const int rcj = run_pitch_jobs(ctx, p->np, pitch_jobs);
        if (rcj) {
            // the new slots were never filled: un-register them, or every later plan would read garbage
            for (size_t i = pitch_job_units.size(); i-- > 0;) p->np->pitch_slots[pitch_job_units[i]].pop_back();
            p->np->pitch_used -= (uint32_t)pitch_jobs.size();
            return rcj;
        }
    }

    // ---- word-region deduplication (run_task in assemble.cuh).  A task is ELIGIBLE when the window it holds on
    // reaching the contour of its first WORD_END is a function of the ops before it alone:
    //   * no MARK before that WORD_END (the region starts with the task), its silence mask fits the shared scratch
    //     (a task longer than the window takes part as well: it is assembled / resumed in place, TASK_GLOBAL);
    //   * every join finds its crossfade / energy window min(xf, n) and its pitch-analysis window min(2 xf, n/2)
    //     inside the region (nothing reaches back into an earlier region), every live fade-out too;
    //   * the remaining count clamps (count >= 200, count / 2 >= analysis window, ctts.c:1983-1987) do not bind,
    //     which holds when the utterance is at least `thresh` samples long at the start of the task (checked on
    //     the device: the first region or two of an utterance usually assemble themselves).
    // Eligible tasks with equal ops (kind, flags, unit / samples, crossfade; the trim flag of the WORD_END) form a
    // group; a group of two or more gets a canonical task that computes the region once per launch.
    struct Dedup { uint32_t w_op = 0, thresh = 0, group = ctts::NO_REGION, whole = ctts::NO_REGION; };
    std::vector<Dedup> dd(ht.size());
    struct Group { uint32_t first_task, count, canon; };
    std::vector<Group> groups;
    if (ctx->knobs.region_dedup) {
        // open-addressing table: 64-bit hash of the signature -> group, equality checked on the ops themselves
        size_t slots = 64;
        while (slots < 2 * ht.size() + 16) slots *= 2;
        std::vector<uint32_t> table(slots, ctts::NO_REGION);
        std::vector<uint64_t> group_hash;
        auto same_ops = [&](uint32_t a0, uint32_t a1, uint32_t b0, uint32_t b1) {   // ops [a0, a1) vs [b0, b1): first 12 bytes, + trim flag of the WORD_END
            if (a1 - a0 != b1 - b0) return false;
            for (uint32_t i = 0; i < a1 - a0; i++)
                if (memcmp(&h_ops[a0 + i - op0], &h_ops[b0 + i - op0], 12) != 0) return false;
            return ((h_ops[a1 - op0].flags ^ h_ops[b1 - op0].flags) & CTTS_WE_TRIM) == 0;
        };
        uint64_t why[4] = {0, 0, 0, 0}, why_bound[4] = {0, 0, 0, 0};   // trace: mask beyond the scratch, reaches back / no WORD_END, (unused), eligible
        for (size_t ti = 0; ti < ht.size(); ti++) {
            const HostTask& h = ht[ti];
            if (h.region_max > scr_samples) { why[0]++; why_bound[0] += h.bound; continue; }
            uint64_t cnt = 0, T = 0, hash = 1469598103934665603ull;
            bool ok = true, found = false;
            uint32_t k = h.op_begin;
            for (; k < h.op_end && ok && !found; k++) {
                const ctts_plan_op& op = h_ops[k - op0];
                switch (op.kind) {
                    case ctts::OP_NOP:
                        break;
                    case CTTS_OP_UNIT: {
                        const uint32_t nu = ucnt[op.a];
                        if (nu == 0) break;
                        if (op.flags & CTTS_UNIT_AFTER_BOUNDARY) { cnt += nu; break; }
                        if (cnt == 0 || op.b == 0) { ok = false; break; }   // joined or not is decided by the count before the region
                        const uint32_t m = std::min(op.b, nu);
                        if (m > cnt) { ok = false; break; }                  // the crossfade would reach back
                        if (nu >= 200) {
                            const uint32_t m2 = 2 * op.b < nu / 2 ? 2 * op.b : nu / 2;   // uint32 like the kernel
                            if (m2 > cnt) { ok = false; break; }             // the pitch analysis would reach back
                            if (2ull * m2 > cnt) T = std::max<uint64_t>(T, 2ull * m2 - cnt);
                            if (200 > cnt) T = std::max<uint64_t>(T, 200 - cnt);
                        }
                        cnt += nu - m;
                        break;
                    }
                    case CTTS_OP_SILENCE:
                        cnt += op.a;
                        break;
                    case CTTS_OP_FADE_OUT:
                        if (op.a > cnt) ok = false;                          // acts on samples of an earlier region
                        break;
                    case CTTS_OP_WORD_END:
                        found = true;
                        break;
                    default:                                                 // MARK before the first WORD_END
                        ok = false;
                }
                if (ok && !found) {   // kind | flags, a, b
                    const uint32_t* wds = reinterpret_cast<const uint32_t*>(&op);
                    hash = (hash ^ wds[0]) * 1099511628211ull;
                    hash = (hash ^ wds[1]) * 1099511628211ull;
                    hash = (hash ^ wds[2]) * 1099511628211ull;
                }
            }
            if (!ok || !found || cnt == 0 || T > 0x7fffffffull) { why[1]++; why_bound[1] += h.bound; continue; }
            why[3]++;
            why_bound[3] += h.bound;
            const uint32_t w = k - 1;
            hash = (hash ^ (h_ops[w - op0].flags & CTTS_WE_TRIM)) * 1099511628211ull;
            hash ^= hash >> 29;
            uint32_t gid = ctts::NO_REGION;
            for (size_t sl = hash & (slots - 1);; sl = (sl + 1) & (slots - 1)) {
                const uint32_t g2 = table[sl];
                if (g2 == ctts::NO_REGION) {
                    gid = (uint32_t)groups.size();
                    table[sl] = gid;
                    groups.push_back(Group{(uint32_t)ti, 0u, ctts::NO_REGION});
                    group_hash.push_back(hash);
                    break;
                }
                if (group_hash[g2] == hash) {
                    const HostTask& f = ht[groups[g2].first_task];
                    if (same_ops(f.op_begin, dd[groups[g2].first_task].w_op, h.op_begin, w)) {
                        gid = g2;
                        break;
                    }
                }
            }
            groups[gid].count++;
            dd[ti].w_op = w;
            dd[ti].thresh = (uint32_t)T;
            dd[ti].group = gid;
        }
        if (ctx->knobs.trace) {
            uint64_t single = 0, single_bound = 0, first = 0, first_bound = 0;
            for (uint32_t ui = 0; ui < n; ui++)
                for (uint32_t ti = ht_begin[ui]; ti < ht_begin[ui + 1]; ti++) {
                    if (dd[ti].group == ctts::NO_REGION) continue;
                    if (groups[dd[ti].group].count < 2) { single++; single_bound += ht[ti].bound; }
                    else if (ti == ht_begin[ui] && dd[ti].thresh) { first++; first_bound += ht[ti].bound; }
                }
            fprintf(stderr, "ctts_gpu: region dedup, %zu tasks: mask beyond the scratch %llu (%llu samples), not a function of their ops %llu (%llu), "
                            "eligible %llu (%llu) of which unique %llu (%llu), first of an utterance with clamps %llu (%llu)\n",
                    ht.size(), (unsigned long long)why[0], (unsigned long long)why_bound[0], (unsigned long long)why[1],
                    (unsigned long long)why_bound[1], (unsigned long long)why[3], (unsigned long long)why_bound[3],
                    (unsigned long long)single, (unsigned long long)single_bound, (unsigned long long)first, (unsigned long long)first_bound);
        }
    }
    // canonical tasks: first in ticket order (an occurrence waits for a SMALLER ticket only), longest first (those
    // longer than the window, the slowest, start first: their occurrences wait the least)
    std::vector<uint32_t> canon_groups;
    for (uint32_t gi = 0; gi < groups.size(); gi++)
        if (groups[gi].count >= 2) canon_groups.push_back(gi);
    std::sort(canon_groups.begin(), canon_groups.end(), [&](uint32_t a, uint32_t b) {
        const uint64_t ba = ht[groups[a].first_task].bound, bb = ht[groups[b].first_task].bound;
        return ba != bb ? ba > bb : a < b;
    });
    const uint32_t n_canon = (uint32_t)canon_groups.size();
    for (uint32_t c = 0; c < n_canon; c++) groups[canon_groups[c]].canon = c;

    // ---- second level: WHOLE tasks that are equal.  A task that resumes from a canonical region and then runs only
    // its WORD_END (trim flag, contour factors, energy ramp -- compared bit for bit) and fade-outs / pauses / marks
    // produces samples that depend on its ops alone (a fade-out that finds fewer samples than it wants reaches back:
    // seen on the device, the result is then not shared).  The first such task in ticket order -- the SOURCE -- also
    // stores what it flushes into the region store; the others (REUSE) copy it from there and run nothing.
    // Row 0 (the utterance is empty when the task starts) can only take part when thresh == 0.
    struct Whole { uint32_t first_task, count, store, row; };
    std::vector<Whole> wholes;
    if (n_canon && ctx->knobs.region_dedup >= 2) {
        size_t slots = 64;
        while (slots < 2 * ht.size() + 16) slots *= 2;
        std::vector<uint32_t> table(slots, ctts::NO_REGION);
        std::vector<uint64_t> whole_hash;
        auto same_tail = [&](size_t ta, size_t tb) {   // the WORD_END in full, the ops behind it like same_ops
            const HostTask& a = ht[ta];
            const HostTask& b = ht[tb];
            if (a.op_end - dd[ta].w_op != b.op_end - dd[tb].w_op) return false;
            if (memcmp(&h_ops[dd[ta].w_op - op0], &h_ops[dd[tb].w_op - op0], sizeof(ctts_plan_op)) != 0) return false;
            for (uint32_t i = 1; i < a.op_end - dd[ta].w_op; i++)
                if (memcmp(&h_ops[dd[ta].w_op + i - op0], &h_ops[dd[tb].w_op + i - op0], 12) != 0) return false;
            return true;
        };
        for (uint32_t ui = 0; ui < n; ui++) {
            for (uint32_t ti = ht_begin[ui]; ti < ht_begin[ui + 1]; ti++) {
                const Dedup& d = dd[ti];
                if (d.group == ctts::NO_REGION || groups[d.group].canon == ctts::NO_REGION) continue;
                if (ti == ht_begin[ui] && d.thresh != 0) continue;
                const HostTask& h = ht[ti];
                uint64_t hash = 1469598103934665603ull ^ d.group;
                bool ok = true;
                for (uint32_t k = d.w_op; k < h.op_end && ok; k++) {
                    const ctts_plan_op& op = h_ops[k - op0];
                    const uint32_t* wds = reinterpret_cast<const uint32_t*>(&op);
                    if (k == d.w_op) {
                        for (int i = 0; i < 8; i++) hash = (hash ^ wds[i]) * 1099511628211ull;
                        continue;
                    }
                    if (op.kind != ctts::OP_NOP && op.kind != CTTS_OP_FADE_OUT && op.kind != CTTS_OP_SILENCE && op.kind != CTTS_OP_MARK) ok = false;
                    for (int i = 0; i < 3; i++) hash = (hash ^ wds[i]) * 1099511628211ull;
                }
                if (!ok) continue;
                hash ^= hash >> 29;
                uint32_t wid = ctts::NO_REGION;
                for (size_t sl = hash & (slots - 1);; sl = (sl + 1) & (slots - 1)) {
                    const uint32_t w2 = table[sl];
                    if (w2 == ctts::NO_REGION) {
                        wid = (uint32_t)wholes.size();
                        table[sl] = wid;
                        wholes.push_back(Whole{ti, 0u, ctts::NO_REGION, 0u});
                        whole_hash.push_back(hash);
                        break;
                    }
                    if (whole_hash[w2] == hash && dd[wholes[w2].first_task].group == d.group && same_tail(wholes[w2].first_task, ti)) {
                        wid = w2;
                        break;
                    }
                }
                wholes[wid].count++;
                dd[ti].whole = wid;
            }
        }
    }

    // ticket order: canonical regions, then region-major (task k of every utterance before task k+1 of any),
    // inside a row longest first (it is the one a successor may have to wait for, and longest-first
    // balances the tail of the launch); tasks that copy a whole task's samples are short and all latency: those whose
    // source sits in an earlier row are spread evenly over the row (an SM then always has contours to issue while a
    // copy waits for memory), those whose source is in the same row close it (and so run well after it)
    std::vector<uint32_t> order;              // ht indices in ticket order
    std::vector<uint32_t> ht_ui(ht.size());
    for (uint32_t ui = 0; ui < n; ui++)
        for (uint32_t ti = ht_begin[ui]; ti < ht_begin[ui + 1]; ti++) ht_ui[ti] = ui;
    order.reserve(ht.size());
    std::vector<uint8_t> is_reuse(ht.size(), 0);
    uint32_t n_sources = 0;
    {
        std::vector<uint32_t> row(n), tail, kept, early;
        for (uint32_t k = 0; k < max_rows; k++) {
            uint32_t m = 0;
            for (uint32_t i = 0; i < n; i++)
                if (k < ht_begin[i + 1] - ht_begin[i]) row[m++] = i;
            std::sort(row.begin(), row.begin() + m, [&](uint32_t a, uint32_t b) {
                const uint64_t ba = ht[ht_begin[a] + k].bound, bb = ht[ht_begin[b] + k].bound;
                return ba != bb ? ba > bb : a < b;
            });
            tail.clear();
            kept.clear();
            early.clear();
            for (uint32_t i = 0; i < m; i++) {
                const uint32_t ti = ht_begin[row[i]] + k;
                const uint32_t w = dd[ti].whole;
                if (w != ctts::NO_REGION && wholes[w].count >= 2) {
                    if (wholes[w].store == ctts::NO_REGION) {
                        wholes[w].store = n_canon + n_sources++;
                        wholes[w].first_task = ti;     // the source
                        wholes[w].row = k;
                    } else {
                        is_reuse[ti] = 1;
                        (wholes[w].row < k ? early : tail).push_back(row[i]);
                        continue;
                    }
                }
                kept.push_back(row[i]);
            }
            size_t ie = 0;
            for (size_t i = 0; i < kept.size(); i++) {
                order.push_back(ht_begin[kept[i]] + k);
                for (const size_t want = (i + 1) * early.size() / kept.size(); ie < want; ie++) order.push_back(ht_begin[early[ie]] + k);
            }
            for (; ie < early.size(); ie++) order.push_back(ht_begin[early[ie]] + k);
            for (uint32_t ui : tail) order.push_back(ht_begin[ui] + k);
        }
    }

    const uint32_t n_store = n_canon + n_sources;
    std::vector<unsigned long long> region_off(n_store + 1, 0);
    for (uint32_t c = 0; c < n_canon; c++)
        region_off[c + 1] = up8(ht[groups[canon_groups[c]].first_task].bound) + 8;
    for (const Whole& w : wholes)
        if (w.store != ctts::NO_REGION) region_off[w.store + 1] = up8(ht[w.first_task].bound) + 8;
    for (uint32_t c = 0; c < n_store; c++) region_off[c + 1] += region_off[c];
    if (region_off.back() >> 3 > 0xffffffffull) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "region store larger than 2^35 samples");
    if (n_store) {
        PlanAlloc al{p, false};
        al.d_used = p->d_used;
        p->d_region_store = al.dev<int16_t>(region_off.back());
        p->d_region_state = al.dev<unsigned long long>(n_store);
        p->d_used = al.d_used;
        if (al.err != cudaSuccess)
            return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "region store");
        CU(ctx, cudaMemsetAsync(p->d_region_state, 0, (size_t)n_store * 8, st));
    }

    uint32_t nt = 0;
    for (uint32_t c = 0; c < canon_groups.size(); c++) {
        const uint32_t ti = groups[canon_groups[c]].first_task;
        const HostTask& h = ht[ti];
        ctts::RegionTask t{};
        t.op_begin = h.op_begin - op0;
        t.op_end = dd[ti].w_op + 1 - op0;
        t.bound = (uint32_t)h.bound;
        t.pred = -1;
        t.flags = ctts::TASK_CANON | (h.bound > wcap ? (uint32_t)ctts::TASK_GLOBAL : 0u);   // assembled in its slot
        t.dst_cap = (uint32_t)(region_off[c + 1] - region_off[c]);
        t.dst_off = region_off[c];
        t.big = 0xffffffffu;
        t.region = c;
        t.whole = ctts::NO_REGION;
        t.w_op = dd[ti].w_op - op0;
        p->h_tasks[nt++] = t;
    }
    p->info.n_canon_tasks = n_canon;
    std::vector<int32_t> last_index(n, -1);
    int build_rc = CTTS_GPU_OK;
    auto make_task = [&](uint32_t hti) {
        const uint32_t u = ht_ui[hti];
        const uint32_t k = hti - ht_begin[u];
        const HostTask& h = ht[hti];
        ctts::RegionTask t{};
        t.utt = u;
        t.op_begin = h.op_begin - op0;
        t.op_end = h.op_end - op0;
        t.bound = (uint32_t)std::min<uint64_t>(h.bound, 0xffffffffull);
        t.pred = last_index[u];
        const bool stretched = p->pre_off[u] != ~0ull;
        t.flags = (k + 1 == ht_begin[u + 1] - ht_begin[u] ? (uint32_t)ctts::TASK_LAST : 0u) | (stretched ? (uint32_t)ctts::TASK_TO_PRE : 0u);
        if (h.bound > wcap) { t.flags |= ctts::TASK_GLOBAL; p->info.n_global_tasks++; }
        t.dst_cap = stretched ? (uint32_t)p->pre_cap[u] : (uint32_t)(p->n_offsets[u + 1] - p->n_offsets[u]);
        t.dst_off = stretched ? p->pre_off[u] : p->n_offsets[u];
        t.big = 0xffffffffu;
        if (h.region_max > scr_samples) {
            if (p->n_big >= p->big_cap) build_rc = fail(ctx, CTTS_GPU_ERR_DEVICE, "internal: trim scratch slots");
            else t.big = p->n_big++;
        }
        t.region = ctts::NO_REGION;
        t.whole = ctts::NO_REGION;
        const Dedup& d = dd[hti];
        // (a first task whose clamps can bind never meets its threshold: it assembles itself)
        if (d.group != ctts::NO_REGION && groups[d.group].canon != ctts::NO_REGION && (k > 0 || d.thresh == 0)) {
            t.region = groups[d.group].canon;
            t.region_at = (uint32_t)(region_off[t.region] >> 3);
            t.thresh = h.base_lb >= d.thresh ? 0u : d.thresh;   // 0: met whatever the predecessor's count turns out to be
            t.w_op = d.w_op - op0;
            p->info.n_dedup_tasks++;
            p->info.dedup_bound_samples += h.bound;
            if (d.whole != ctts::NO_REGION && wholes[d.whole].store != ctts::NO_REGION) {
                t.whole = wholes[d.whole].store;
                t.whole_at = (uint32_t)(region_off[t.whole] >> 3);
                if (is_reuse[hti]) {
                    t.flags |= ctts::TASK_REUSE;
                    p->info.n_reuse_tasks++;
                    p->info.reuse_bound_samples += h.bound;
                } else {
                    t.flags |= ctts::TASK_SOURCE;
                    p->info.n_source_tasks++;
                }
            }
        }
        return t;
    };
    for (size_t oi = 0; oi < order.size(); oi++) {
        p->h_tasks[nt] = make_task(order[oi]);
        last_index[ht_ui[order[oi]]] = (int32_t)nt;
        nt++;
    }
    if (build_rc) return build_rc;
    p->n_tasks = nt;
    p->grid = (uint32_t)std::min<uint64_t>((uint64_t)p->occ * (uint64_t)ctx->sm_count, std::max<uint32_t>(nt, 1));
    p->info.n_tasks = nt;
    p->info.grid = p->grid;
    if (n_ops) CU(ctx, cudaMemcpyAsync(p->d_ops, h_ops, (size_t)n_ops * sizeof(ctts_plan_op), cudaMemcpyHostToDevice, st));
    if (nt) CU(ctx, cudaMemcpyAsync(p->d_tasks, p->h_tasks, (size_t)nt * sizeof(ctts::RegionTask), cudaMemcpyHostToDevice, st));
    if (!p->arena) {
        // pageable staging must outlive the async copies
        CU(ctx, cudaStreamSynchronize(st));
        std::vector<char>().swap(p->h_staging);
    }
    return CTTS_GPU_OK;
}
#undef CUP

// Enqueues kernels on one stream, checks each launch and counts it.  A counting Launch enqueues nothing: run over a
// plan's launch code, it gives the plan's kernel_launches.
struct Launch {
    ctts_gpu_ctx* ctx;
    cudaStream_t st;
    bool count_only = false;
    uint32_t count = 0;

    template <class... P, class... A>
    int operator()(void (*kernel)(P...), dim3 grid, uint32_t threads, size_t smem, A... args) {
        count++;
        if (count_only) return CTTS_GPU_OK;
        kernel<<<grid, threads, smem, st>>>(args...);
        CU(ctx, cudaGetLastError());
        return CTTS_GPU_OK;
    }
};

// Rows 0 .. n - 1 of a launch cut into grid.y slices: slice(first row, rows) for each, up to the first error.
template <class F>
int grid_y_slices(uint32_t n, F slice) {
    constexpr uint32_t kMaxGridY = 65535;
    for (uint32_t r0 = 0; r0 < n; r0 += kMaxGridY)
        if (const int rc = slice(r0, std::min(n - r0, kMaxGridY))) return rc;
    return CTTS_GPU_OK;
}

// Enqueue the plan's assembly kernel.  A plan without tasks skips the launch but counts it all the same: the assembly
// kernel is part of every plan's kernel_launches, an empty plan's 1 included.
int launch_assemble(Launch& launch, ctts_gpu_plan* p, int16_t* d_pcm_out) {
    if (p->n_tasks == 0) {
        launch.count++;
        return CTTS_GPU_OK;
    }
    const ctts_gpu_ctx* ctx = launch.ctx;
    ctts::AsmArgs a{};
    a.pool = p->np->d_pool;
    a.unit_meta = p->np->d_meta;
    a.unit_pitch = p->np->d_pitch;
    a.unit_off = ctx->d_unit_off;
    a.unit_cnt = ctx->d_unit_cnt;
    a.n_units = ctx->n_units;
    a.tab.fade_out = ctx->d_tables;
    a.tab.fade_in = ctx->d_tables + 1024;
    a.tab.sine = ctx->d_tables + 2048;
    a.tab.hann256 = ctx->d_tables + 3072;
    a.tab.hann512 = ctx->d_tables + 3328;
    a.tab.xfade4 = reinterpret_cast<const float4*>(ctx->d_tables + 3840);
    a.ops = p->d_ops;
    a.tasks = p->d_tasks;
    a.n_tasks = p->n_tasks;
    a.dst_final = d_pcm_out;
    a.dst_pre = p->d_pre;
    a.out_counts = p->d_counts;
    a.pre_counts = p->d_pre_counts;
    a.err = p->d_err;
    a.trim_scratch = p->d_trim;
    a.trim_scratch_words = p->trim_words;
    a.region_store = p->d_region_store;
    a.region_state = p->d_region_state;
    a.chain = p->d_chain;
    a.ticket = p->d_ticket;
    a.prof = p->d_prof;
    a.epoch = p->epoch;
    a.prm = p->prm;
    a.wcap = p->wcap;
    a.hcap = p->hcap;
    return launch(ctts::assemble_kernel, p->grid, ctts::ASM_THREADS, p->smem_bytes, a);
}

int begin_run(ctts_gpu_ctx* ctx, ctts_gpu_plan* p) {
    cudaStream_t st = ctx->stream;
    CU(ctx, cudaMemsetAsync(p->d_counts, 0, (size_t)p->n_utts * 4, st));
    CU(ctx, cudaMemsetAsync(p->d_pre_counts, 0, (size_t)p->n_utts * 4, st));
    CU(ctx, cudaMemsetAsync(p->d_err, 0, (size_t)p->n_utts * 4, st));
    CU(ctx, cudaMemsetAsync(p->d_ticket, 0, 4, st));
    p->epoch++;
    if (p->epoch == 0) p->epoch = 1;   // (2^32 runs later) the chain words of the last lap are long gone
    return CTTS_GPU_OK;
}

// Enqueue the WSOLA kernels of the plan's stretched utterances (after its assembly kernel).
int launch_stretch(Launch& launch, ctts_gpu_plan* p, int16_t* d_pcm_out) {
    const uint32_t ns = p->n_stretch;
    if (!ns) return CTTS_GPU_OK;
    const ctts_gpu_ctx* ctx = launch.ctx;
    ctts::WsolaArgs w{};
    w.tasks = p->d_stasks;
    w.n_tasks = ns;
    w.pre = p->d_pre;
    w.pre_counts = p->d_pre_counts;
    w.out = d_pcm_out;
    w.out_counts = p->d_counts;
    w.frame_pos = p->d_frame_pos;
    w.n_frames = p->d_n_frames;
    w.first_bad = p->d_n_frames + 2 * (size_t)p->n_stretch;
    w.first_silent = p->d_n_frames + 3 * (size_t)p->n_stretch;
    w.tier2 = p->d_n_frames + 4 * (size_t)p->n_stretch;
    w.task_count = ns;
    w.speculate = ctx->knobs.wsola_speculate ? 1u : 0u;
    w.force_bad = ctx->knobs.wsola_force_bad;
    w.hann512 = ctx->d_tables + 3328;
    w.ola_block_task = p->d_ola_task;
    w.ola_block_first = p->d_ola_first;
    // speculate (scan) -> verify every frame in parallel -> walk the chain only where that failed -> overlap-add
    int rc = launch(ctts::wsola_scan_kernel, (ns + 7) / 8, 256, 0, w);
    if (!rc && w.speculate && p->verify_tiles)
        rc = grid_y_slices(ns, [&](uint32_t t0, uint32_t rows) {
            ctts::WsolaArgs wv = w;
            wv.task_first = t0;
            return launch(ctts::wsola_verify_kernel, dim3(p->verify_tiles, rows), ctts::WV_THREADS, sizeof(ctts::WvSmem), wv);
        });
    if (!rc) rc = launch(ctts::wsola_search_kernel, ns, ctts::WS_THREADS, 0, w);
    if (!rc && p->n_ola_blocks) rc = launch(ctts::wsola_ola_kernel, p->n_ola_blocks, ctts::OLA_THREADS, 0, w);
    return rc;
}

// Enqueue the output-rate conversion of the plan (after its WSOLA kernels): native slots d_nat and
// counts -> output-rate slots d_final and d_rs_counts.  Nothing at the native rate.
int launch_resample(Launch& launch, ctts_gpu_plan* p, const int16_t* d_nat, int16_t* d_final) {
    const ctts_gpu_ctx::RsTable* rs = p->rs;
    if (!rs || !p->n_utts) return CTTS_GPU_OK;
    const uint32_t n = p->n_utts;
    return grid_y_slices(n, [&](uint32_t u0, uint32_t rows) {
        ctts::ResampleArgs r{};
        r.in = d_nat;
        r.in_off = p->d_off + u0;
        r.in_counts = p->d_counts + u0;
        r.out = d_final;
        r.out_off = slot_off(p) + u0;
        r.out_counts = p->d_rs_counts + u0;
        r.taps = reinterpret_cast<const float4*>(rs->d_taps);
        r.L = rs->L;
        r.M = rs->M;
        r.kp = rs->kp;
        r.c = rs->c;
        r.smem_floats = rs->smem_floats;
        return launch(ctts::resample_kernel, dim3(p->rs_tiles, rows), ctts::RS_THREADS, rs->smem_floats * sizeof(float), r);
    });
}

// Enqueue the loudness normalization of the plan (after its output-rate conversion), in place on the output-rate
// slots d_final.  Nothing when the stage is off.
int launch_loudness(Launch& launch, ctts_gpu_plan* p, int16_t* d_final) {
    const ctts_gpu_ctx::LdTable* ld = p->ld;
    if (!ld || !p->n_utts) return CTTS_GPU_OK;
    const uint32_t n = p->n_utts;
    ctts::LdArgs a{};
    a.pcm = d_final;
    a.off = slot_off(p);
    a.counts = p->d_final_counts;
    a.state = p->d_ld_state;
    a.energy = p->d_ld_energy;
    a.peak = p->d_ld_peak;
    a.lufs = p->d_ld_lufs;
    a.gain = p->d_ld_gain;
    a.table = launch.ctx->d_ld_gains;
    a.gate_abs = pow(10.0, (-70.0 + 0.691) / 10.0);
    a.n = n;
    a.ceiling = ld->ceiling_q;
    a.target = ld->target;
    a.f = ld->f;
    if (ld->true_peak) {
        a.tp_tile = p->d_ld_tp_tile;
        a.tp_peak = p->d_ld_tp;
        memcpy(a.tp_h, ld->tp_h, sizeof a.tp_h);
    }
    auto sliced = [&](auto kernel, uint32_t tiles, uint32_t threads) {
        const int rc = grid_y_slices(n, [&](uint32_t u0, uint32_t rows) {
            a.u0 = u0;
            return launch(kernel, dim3(tiles, rows), threads, 0, a);
        });
        a.u0 = 0;
        return rc;
    };
    int rc = sliced(ctts::ld_chunk_kernel<false>, p->ld_tiles, ctts::LD_THREADS);
    if (!rc) rc = launch(ctts::ld_scan_kernel, (n + ctts::LD_SCAN_THREADS - 1) / ctts::LD_SCAN_THREADS, ctts::LD_SCAN_THREADS, 0, a);
    if (!rc) rc = sliced(ctts::ld_chunk_kernel<true>, p->ld_tiles, ctts::LD_THREADS);
    if (!rc && ld->true_peak) rc = sliced(ctts::ld_true_peak_kernel, p->ld_tp_tiles, ctts::LD_TP_THREADS);
    if (!rc) rc = launch(ld->true_peak ? ctts::ld_gain_kernel<true> : ctts::ld_gain_kernel<false>, n, ctts::LD_GAIN_THREADS, 0, a);
    return rc ? rc : sliced(ctts::ld_apply_kernel, p->ld_apply_tiles, ctts::LD_APPLY_THREADS);
}

// Enqueue the plan's stage chain: assembly and WSOLA into the native-rate slots d_nat, output-rate conversion into
// d_final (the same slots at the native rate), loudness normalization in place there.
int launch_chain(Launch& launch, ctts_gpu_plan* p, int16_t* d_nat, int16_t* d_final) {
    int rc = launch_assemble(launch, p, d_nat);
    if (!rc) rc = launch_stretch(launch, p, d_nat);
    if (!rc) rc = launch_resample(launch, p, d_nat, d_final);
    return rc ? rc : launch_loudness(launch, p, d_final);
}

}  // namespace

extern "C" {

int ctts_gpu_plan_create(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, const ctts_assembly_params* params,
                         const uint64_t* out_offsets, ctts_gpu_plan** out) {
    ctts_gpu_plan* p = nullptr;
    int rc = prepare_plan(ctx, plan, params, out_offsets, nullptr, &p);
    if (!rc) rc = build_tasks(ctx, p, plan, ctx->stream);
    if (rc) {
        ctts_gpu_plan_destroy(p);
        return rc;
    }
    Launch count{ctx, ctx->stream, true};
    launch_chain(count, p, nullptr, nullptr);   // (launches nothing: cannot fail)
    p->info.kernel_launches = count.count;
    *out = p;
    return CTTS_GPU_OK;
}

uint64_t ctts_gpu_plan_out_samples(const ctts_gpu_plan* p) { return p ? p->offsets[p->n_utts] : 0; }

int ctts_gpu_plan_out_offsets(const ctts_gpu_plan* p, uint64_t* offsets) {
    if (!p || !offsets) return CTTS_GPU_ERR_INVALID_ARG;
    std::copy(p->offsets.begin(), p->offsets.end(), offsets);
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_info(const ctts_gpu_plan* p, ctts_gpu_run_info* info) {
    if (!p || !info) return CTTS_GPU_ERR_INVALID_ARG;
    *info = p->info;
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_run(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, int16_t* d_pcm_out) {
    if (!ctx || !p || p->ctx != ctx) return CTTS_GPU_ERR_INVALID_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    if (!d_pcm_out) {
        if (!p->d_out_owned)
            CU(ctx, cudaMalloc(reinterpret_cast<void**>(&p->d_out_owned),
                               std::max<uint64_t>(p->offsets[p->n_utts], 8) * sizeof(int16_t)));
        d_pcm_out = p->d_out_owned;
    }
    p->d_out_last = d_pcm_out;
    if (p->n_utts == 0) return CTTS_GPU_OK;
    int16_t* d_nat = d_pcm_out;   // where the assembly and WSOLA kernels write
    if (p->rs) {
        if (!p->d_nat_owned)
            CU(ctx, cudaMalloc(reinterpret_cast<void**>(&p->d_nat_owned), std::max<uint64_t>(p->n_offsets[p->n_utts], 8) * sizeof(int16_t)));
        d_nat = p->d_nat_owned;
    }
    Launch launch{ctx, ctx->stream};
    const int rc = begin_run(ctx, p);
    return rc ? rc : launch_chain(launch, p, d_nat, d_pcm_out);
}

int ctts_gpu_plan_read_counts(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, uint32_t* out_counts) {
    if (!ctx || !p || !out_counts) return CTTS_GPU_ERR_INVALID_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    if (p->n_utts == 0) return CTTS_GPU_OK;
    std::vector<uint32_t> err(p->n_utts);
    CU(ctx, cudaMemcpyAsync(out_counts, p->d_final_counts, (size_t)p->n_utts * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(err.data(), p->d_err, (size_t)p->n_utts * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t u = 0; u < p->n_utts; u++)
        if (err[u]) return fail(ctx, CTTS_GPU_ERR_DEVICE, "utterance %u: device error %u", u, err[u]);
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_read_pcm(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, int16_t* dst, uint64_t first, uint64_t n) {
    if (!ctx || !p || !dst || !p->d_out_last || first + n > p->offsets[p->n_utts]) return CTTS_GPU_ERR_INVALID_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst, p->d_out_last + first, n * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_read_loudness(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, double* lufs, uint32_t* gain) {
    if (!ctx || !p || p->ctx != ctx || !lufs || !gain) return CTTS_GPU_ERR_INVALID_ARG;
    if (!p->ld) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "the plan was created with loudness normalization off");
    if (p->n_utts == 0) return CTTS_GPU_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(lufs, p->d_ld_lufs, (size_t)p->n_utts * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(gain, p->d_ld_gain, (size_t)p->n_utts * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_read_true_peak(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, float* peak) {
    if (!ctx || !p || p->ctx != ctx || !peak) return CTTS_GPU_ERR_INVALID_ARG;
    if (!p->ld || !p->ld->true_peak) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "the plan was not created with a true-peak ceiling");
    if (p->n_utts == 0) return CTTS_GPU_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(peak, p->d_ld_tp, (size_t)p->n_utts * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_wsola_stats(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, ctts_gpu_wsola_stats* out) {
    if (!ctx || !p || !out) return CTTS_GPU_ERR_INVALID_ARG;
    memset(out, 0, sizeof *out);
    if (!p->n_stretch) return CTTS_GPU_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t ns = p->n_stretch;
    std::vector<uint32_t> h(5 * ns);
    CU(ctx, cudaMemcpyAsync(h.data(), p->d_n_frames, h.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < ns; i++) {
        const uint32_t frames = h[i], bad = h[2 * ns + i];
        out->frames += frames;
        out->exact_evaluations += h[ns + i];
        out->tier2_candidates += h[4 * ns + i];
        if (bad < frames) {
            out->walked_utterances++;
            out->walked_frames += frames - bad;
        }
    }
    return CTTS_GPU_OK;
}

int ctts_gpu_plan_read_pre(ctts_gpu_ctx* ctx, ctts_gpu_plan* p, uint32_t u, int16_t* dst, uint64_t cap, uint64_t* n) {
    if (!ctx || !p || !dst || !n || u >= p->n_utts || p->pre_off[u] == ~0ull) return CTTS_GPU_ERR_INVALID_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    uint32_t cnt = 0;
    CU(ctx, cudaMemcpyAsync(&cnt, p->d_pre_counts + u, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    *n = cnt;
    uint64_t take = std::min<uint64_t>(cnt, cap);
    CU(ctx, cudaMemcpy(dst, p->d_pre + p->pre_off[u], take * sizeof(int16_t), cudaMemcpyDeviceToHost));
    return CTTS_GPU_OK;
}

// ---------------------------------------------------------------- sessions: a batch fed in pieces

}  // extern "C"

// What a session delivers: PCM samples, or bytes (one FLAC file per utterance, or one G.711 code per sample)
enum SessionOutput { OUT_PCM = 0, OUT_ULAW = CTTS_GPU_G711_ULAW, OUT_ALAW = CTTS_GPU_G711_ALAW, OUT_FLAC };
static_assert(OUT_ULAW == ctts::G711_ULAW && OUT_ALAW == ctts::G711_ALAW, "G.711 law constants");

// What the delivery path needs to know of each output kind, indexed by SessionOutput
struct OutputKind {
    uint32_t unit_bytes;   // host bytes of one unit: capacity, cursor and offsets count units
    uint32_t align;        // a packed utterance takes its size rounded up to this many units
    const char *unit, *name, *submit;   // for error messages: the units, the kind, the submit call it takes
};
constexpr OutputKind kOutput[] = {{2, 8, "samples", "PCM", "ctts_gpu_session_submit"},
                                  {1, 8, "bytes", "G.711", "ctts_gpu_session_submit_g711"},
                                  {1, 8, "bytes", "G.711", "ctts_gpu_session_submit_g711"},
                                  {1, 16, "bytes", "FLAC", "ctts_gpu_session_submit_flac"}};

// Where a piece of n utterances keeps its results.  h_res (pinned, 4-byte words): counts [n], device error flags [n],
// (FLAC: file bytes [n], then, 8-byte aligned, the first frame descriptor of every utterance [n + 1]).  FLAC uploads
// those frame bases to d_pack_off behind the n + 1 packed offsets.
struct ResLayout {
    size_t flags, bytes, size, bases;          // word offsets in h_res; size: what sizes a packed utterance
    size_t base_words, res_words, off_words;   // 8-byte words at bases; the words h_res and d_pack_off need
    ResLayout(uint32_t n, SessionOutput k) : flags(n), bytes(2 * (size_t)n) {
        const size_t heads = k == OUT_FLAC ? 3 : 2;
        size = k == OUT_FLAC ? bytes : 0;   // the file bytes, else the count
        bases = (heads * n + 1) & ~(size_t)1;
        base_words = k == OUT_FLAC ? (size_t)n + 1 : 0;
        res_words = bases + 2 + 2 * base_words;
        off_words = (size_t)n + 1 + base_words;
    }
};

struct ctts_gpu_session {
    ctts_gpu_ctx* ctx;
    ctts_assembly_params prm;
    SessionOutput kind;
    uint8_t* out;                 // the caller's buffer
    uint64_t capacity;            // units of kOutput[kind]
    ctts_gpu_chunk_fn on_piece;
    void* user;
    std::chrono::steady_clock::time_point t0;
    uint64_t cursor = 0;          // next free unit (library-chosen layout)
    uint32_t submitted = 0, harvested = 0;   // pieces
    uint32_t copy_next = 0;       // packed mode: first piece whose copy is not enqueued yet
    uint32_t utts = 0;            // utterances submitted so far
    int error = 0;
    uint64_t d2h_bytes = 0;       // copied to the host
};

namespace {

void drain(ctts_gpu_ctx* ctx) {
    cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
}

// Packed mode: the counts of the lane's piece are (or will shortly be) on the host; lay its utterances out
// back to back at the session's cursor and enqueue ONE copy of exactly the units that exist.
int enqueue_packed_copy(ctts_gpu_session* s, ctts_gpu_ctx::Lane& l) {
    ctts_gpu_ctx* ctx = s->ctx;
    const OutputKind& k = kOutput[s->kind];
    l.copy_pending = false;
    cudaError_t e = cudaEventSynchronize(l.counts_ready);
    if (e != cudaSuccess) {
        if (!s->error) s->error = fail(ctx, CTTS_GPU_ERR_CUDA, "piece of utterances %u..%u: %s", l.utt_base, l.utt_base + l.n, cudaGetErrorString(e));
        return s->error;
    }
    const uint32_t* h_size = l.h_res + ResLayout(l.n, s->kind).size;
    uint64_t o = s->cursor;
    for (uint32_t u = 0; u < l.n; u++) {
        if (l.user_offsets) l.user_offsets[u] = o;
        o += (h_size[u] + (k.align - 1ull)) & ~(k.align - 1ull);
    }
    const uint64_t len = o - s->cursor;
    if (o > s->capacity) {
        if (!s->error) s->error = fail(ctx, CTTS_GPU_ERR_BOUNDS, "output buffer too small: %llu %s needed up to utterance %u", (unsigned long long)o, k.unit, l.utt_base + l.n);
        return s->error;
    }
    if (len) e = cudaMemcpyAsync(s->out + s->cursor * k.unit_bytes, l.d_pack, len * k.unit_bytes, cudaMemcpyDeviceToHost, ctx->copy_stream);
    if (e == cudaSuccess) e = cudaEventRecord(l.copied, ctx->copy_stream);
    if (e != cudaSuccess) {
        if (!s->error) s->error = fail(ctx, CTTS_GPU_ERR_CUDA, "D2H: %s", cudaGetErrorString(e));
        return s->error;
    }
    s->d2h_bytes += len * k.unit_bytes;
    s->cursor = o;
    return CTTS_GPU_OK;
}

// Packed mode: enqueue, in order, the copies of the pieces whose counts have arrived; pieces up to and
// including `must` (a piece index, or none: 0xffffffff... never) are waited for.  Keeps the copy stream fed
// while the host is about to block on an older piece.
void pump_copies(ctts_gpu_session* s, uint32_t must_upto) {
    ctts_gpu_ctx* ctx = s->ctx;
    while (s->copy_next < s->submitted) {
        ctts_gpu_ctx::Lane& c = ctx->lane[s->copy_next % ctts_gpu_ctx::kLanes];
        if (c.busy && c.copy_pending) {
            if (s->copy_next >= must_upto && cudaEventQuery(c.counts_ready) != cudaSuccess) break;
            enqueue_packed_copy(s, c);
        }
        s->copy_next++;
    }
}

// Wait for the oldest piece in flight, hand its counts (and the piece itself) to the caller, free its lane.
int harvest_one(ctts_gpu_session* s) {
    ctts_gpu_ctx* ctx = s->ctx;
    ctts_gpu_ctx::Lane& l = ctx->lane[s->harvested % ctts_gpu_ctx::kLanes];
    pump_copies(s, s->harvested + 1);   // this piece's copy for sure, and every later one that is ready
    s->harvested++;
    if (!l.busy) return CTTS_GPU_OK;
    int rc = s->error;
    cudaError_t e = cudaEventSynchronize(l.copied);
    if (e != cudaSuccess && !rc) rc = fail(ctx, CTTS_GPU_ERR_CUDA, "piece of utterances %u..%u: %s", l.utt_base, l.utt_base + l.n, cudaGetErrorString(e));
    if (!rc) {
        const ResLayout r(l.n, s->kind);
        const uint32_t* h_err = l.h_res + r.flags;
        if (l.user_counts) memcpy(l.user_counts, l.h_res, (size_t)l.n * 4);
        if (l.user_bytes) memcpy(l.user_bytes, l.h_res + r.bytes, (size_t)l.n * 4);
        for (uint32_t u = 0; u < l.n && !rc; u++)
            if (h_err[u]) rc = fail(ctx, CTTS_GPU_ERR_DEVICE, "utterance %u: device error %u", l.utt_base + u, h_err[u]);
    }
    if (ctx->knobs.trace)
        fprintf(stderr, "  piece of utterances %u..%u on the host at %.1f ms\n", l.utt_base, l.utt_base + l.n,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - s->t0).count());
    // a piece with a device error is not handed over (its counts are arbitrary)
    if (!rc && !s->error && s->on_piece && l.n) s->on_piece(s->user, l.utt_base, l.utt_base + l.n);
    if (rc && !s->error) s->error = rc;
    if (l.plan) {
        if (rc) drain(ctx);
        ctts_gpu_plan_destroy(l.plan);
        l.plan = nullptr;
    }
    l.busy = false;
    return rc;
}

// Grow-only device buffer: at least `bytes` afterwards, *cap in bytes.  zero: a new allocation is zero-filled on the
// context's stream, so that bytes no kernel writes do not carry an earlier allocation's to the host.
template <class T>
int grow(ctts_gpu_ctx* ctx, T** buf, uint64_t* cap, uint64_t bytes, bool zero, const char* what) {
    if (bytes <= *cap) return CTTS_GPU_OK;
    cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    const uint64_t c = bytes + bytes / 8 + 32768;
    if (cudaMalloc(reinterpret_cast<void**>(buf), c) != cudaSuccess)
        return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "%s of %llu bytes", what, (unsigned long long)c);
    if (zero && cudaMemsetAsync(*buf, 0, c, ctx->stream) != cudaSuccess) return fail(ctx, CTTS_GPU_ERR_CUDA, "memset");
    *cap = c;
    return CTTS_GPU_OK;
}

// FLAC frames of the slot of utterance u
uint64_t slot_frames(const ctts_gpu_plan* p, uint32_t u) { return (p->offsets[u + 1] - p->offsets[u] + ctts::FLAC_BLOCK - 1) / ctts::FLAC_BLOCK; }

// Grow the lane's workspace for the piece p: slots, packed output and offsets, pinned results.
int grow_lane(ctts_gpu_session* s, ctts_gpu_ctx::Lane& l, const ctts_gpu_plan* p, bool packed) {
    ctts_gpu_ctx* ctx = s->ctx;
    const uint32_t n = p->n_utts;
    const uint64_t total = p->offsets[n];
    const ResLayout r(n, s->kind);
    int rc = grow(ctx, &l.d_out, &l.d_out_cap, p->n_offsets[n] * sizeof(int16_t), true, "output slots");
    if (!rc && p->rs) rc = grow(ctx, &l.d_rs, &l.d_rs_cap, total * sizeof(int16_t), true, "output-rate slots");
    uint64_t pack_bytes = total * kOutput[s->kind].unit_bytes;
    if (s->kind == OUT_FLAC) {   // files and frame descriptors are sized by the slots (>= the bounds): ctts_gpu_flac_bound each
        uint64_t frames = 0;
        pack_bytes = 0;
        for (uint32_t u = 0; u < n; u++) {
            frames += slot_frames(p, u);
            pack_bytes += (ctts_gpu_flac_bound(p->offsets[u + 1] - p->offsets[u]) + 15) & ~15ull;
        }
        if (!rc) rc = grow(ctx, &l.d_frames, &l.d_frames_cap, frames * sizeof(ctts::FlacFrame), false, "FLAC frames");
        if (!rc) rc = grow(ctx, &l.d_flac_info, &l.d_flac_info_cap, 3 * (uint64_t)n * 4, false, "FLAC sizes");
    }
    if (!rc && packed) rc = grow(ctx, &l.d_pack, &l.d_pack_cap, pack_bytes, true, "packed output");
    if (!rc && packed) rc = grow(ctx, &l.d_pack_off, &l.d_pack_off_cap, r.off_words * 8, false, "pack offsets");
    if (rc) return rc;
    if (r.res_words > l.h_res_cap) {
        if (l.h_res) cudaFreeHost(l.h_res);
        l.h_res = nullptr;
        l.h_res_cap = 0;
        const size_t cap = r.res_words + 4096;
        if (cudaHostAlloc(reinterpret_cast<void**>(&l.h_res), cap * 4, cudaHostAllocDefault) != cudaSuccess)
            return fail(ctx, CTTS_GPU_ERR_OUT_OF_MEMORY, "pinned counts");
        l.h_res_cap = cap;
    }
    return CTTS_GPU_OK;
}

// Packed mode: encode the piece's output-rate slots d_final into d_pack, its utterances back to back.  The scan kernel
// stores the counts and flags (FLAC: and file sizes) straight into h_res; counts_ready is recorded behind it, and the
// copy to the caller is enqueued once they are on the host.
int encode_packed(Launch& launch, ctts_gpu_session* s, ctts_gpu_ctx::Lane& l, const ctts_gpu_plan* p, const int16_t* d_final) {
    ctts_gpu_ctx* ctx = s->ctx;
    const cudaStream_t st = launch.st;
    const uint32_t n = p->n_utts;
    const uint32_t* const cnt = p->d_final_counts;
    const unsigned long long* const d_slot = slot_off(p);
    uint64_t max_slot = 0;
    for (uint32_t u = 0; u < n; u++) max_slot = std::max<uint64_t>(max_slot, p->offsets[u + 1] - p->offsets[u]);
    // PCM and G.711: device prefix sum of the counts -> packed positions -> `kernel` copies or encodes every
    // utterance there, padding included
    auto pack = [&](auto kernel, auto* dst) {
        int rc = launch(ctts::pack_scan_kernel, 1, 1024, 0, cnt, p->d_err, n, l.d_pack_off, l.h_res);
        if (rc) return rc;
        CU(ctx, cudaEventRecord(l.counts_ready, st));   // counts and flags are on the host
        const uint32_t tiles = (uint32_t)((max_slot + ctts::PACK_TILE - 1) / ctts::PACK_TILE);
        return grid_y_slices(n, [&](uint32_t u0, uint32_t rows) {
            return launch(kernel, dim3(tiles, rows), ctts::PACK_THREADS, 0, d_final, d_slot + u0, cnt + u0, l.d_pack_off + u0, dst);
        });
    };
    switch (s->kind) {
    case OUT_PCM: return pack(ctts::pack_copy_kernel, reinterpret_cast<int16_t*>(l.d_pack));
    case OUT_ULAW: return pack(ctts::g711_pack_kernel<ctts::G711_ULAW>, l.d_pack);
    case OUT_ALAW: return pack(ctts::g711_pack_kernel<ctts::G711_ALAW>, l.d_pack);
    case OUT_FLAC: break;
    }
    // FLAC: the first frame descriptor of every utterance goes behind the packed offsets; analyse every frame -> sizes
    // and packed byte offsets (counts, flags and sizes into h_res) -> emit each frame at its offset
    unsigned long long* const h_base = reinterpret_cast<unsigned long long*>(l.h_res + ResLayout(n, s->kind).bases);
    unsigned long long* const d_base = l.d_pack_off + (n + 1);
    h_base[0] = 0;
    for (uint32_t u = 0; u < n; u++) h_base[u + 1] = h_base[u] + slot_frames(p, u);
    CU(ctx, cudaMemcpyAsync(d_base, h_base, ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, st));
    const ctts::FlacArgs fa{d_final, d_slot, cnt, d_base, l.d_frames, l.d_pack_off, l.d_flac_info, l.d_pack,
                            p->rs ? p->rs->hz : (uint32_t)CTTS_PLAN_SAMPLE_RATE};
    const uint32_t frames = (uint32_t)std::max<uint64_t>((max_slot + ctts::FLAC_BLOCK - 1) / ctts::FLAC_BLOCK, 1);
    auto frame_grid = [&](auto kernel) {
        return grid_y_slices(n, [&](uint32_t u0, uint32_t rows) { return launch(kernel, dim3(frames, rows), ctts::FLAC_THREADS, 0, fa, u0); });
    };
    int rc = frame_grid(ctts::flac_analyze_kernel);
    if (!rc) rc = launch(ctts::flac_scan_kernel, 1, 1024, 0, fa, p->d_err, n, l.h_res);
    if (rc) return rc;
    CU(ctx, cudaEventRecord(l.counts_ready, st));   // counts, flags and sizes are on the host
    return frame_grid(ctts::flac_emit_kernel);
}

// Slot mode: copy the piece from the device slots (packed by their bounds, up8(bound) + 8 each) to the caller's
// (runs of utterances whose host slots are laid out the same way go in one copy), then its counts and flags to h_res.
cudaError_t copy_slots(ctts_gpu_session* s, ctts_gpu_ctx::Lane& l, const ctts_gpu_plan* p, const int16_t* d_final,
                       const uint64_t* slot_off, const uint64_t* slot_cap) {
    const cudaStream_t cs = s->ctx->copy_stream;
    const uint32_t n = p->n_utts;
    const std::vector<uint64_t>& o = p->offsets;
    cudaError_t e = cudaSuccess;
    for (uint32_t u = 0; u < n && e == cudaSuccess;) {
        uint32_t v = u;
        while (v + 1 < n && slot_off[v + 1] == slot_off[v] + (o[v + 1] - o[v]) && slot_cap[v] >= o[v + 1] - o[v]) v++;
        const uint64_t len = (o[v] - o[u]) + std::min<uint64_t>(o[v + 1] - o[v], slot_cap[v]);
        if (len) e = cudaMemcpyAsync(s->out + slot_off[u] * sizeof(int16_t), d_final + o[u], len * sizeof(int16_t), cudaMemcpyDeviceToHost, cs);
        s->d2h_bytes += len * sizeof(int16_t);
        u = v + 1;
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(l.h_res, p->d_final_counts, (size_t)n * 4, cudaMemcpyDeviceToHost, cs);
    if (e == cudaSuccess) e = cudaMemcpyAsync(l.h_res + ResLayout(n, s->kind).flags, p->d_err, (size_t)n * 4, cudaMemcpyDeviceToHost, cs);
    if (e == cudaSuccess) e = cudaEventRecord(l.copied, cs);
    return e;
}

// One piece: compile, launch, copy.  Utterance i of the piece is delivered to the caller's buffer at slot_off[i],
// slot_cap[i] samples of room (>= its bound); slot_off == nullptr (FLAC and G.711 always): the library appends packed
// slots at the session's cursor and reports them through offsets_out (FLAC: and the file sizes through out_bytes).
// Asynchronous: returns once everything is enqueued.
int submit_piece(ctts_gpu_session* s, const ctts_batch_plan* piece, const uint64_t* slot_off, const uint64_t* slot_cap,
                 uint64_t* offsets_out, uint32_t* out_counts, uint32_t* out_bytes = nullptr) {
    ctts_gpu_ctx* ctx = s->ctx;
    const uint32_t n = piece->n_utts;
    ctts_gpu_ctx::Lane& l = ctx->lane[s->submitted % ctts_gpu_ctx::kLanes];
    const auto tsub0 = std::chrono::steady_clock::now();
    if (s->submitted - s->harvested >= (uint32_t)ctts_gpu_ctx::kLanes) harvest_one(s);   // the lane's previous piece
    if (s->error) return s->error;
    const auto tp0 = std::chrono::steady_clock::now();
    ctts_gpu_plan* p = nullptr;
    int rc = prepare_plan(ctx, piece, &s->prm, nullptr, &l.arena, &p);
    if (rc) return rc;
    const auto tp1 = std::chrono::steady_clock::now();
    auto bail = [&](int code) {
        drain(ctx);
        ctts_gpu_plan_destroy(p);
        return code;
    };
    const bool packed = slot_off == nullptr;   // library layout: exactly the samples that exist, back to back
    for (uint32_t u = 0; u < n && !packed; u++)
        if ((slot_off[u] & 7) || slot_cap[u] < p->bounds[u] || slot_off[u] + slot_cap[u] > s->capacity)
            return bail(fail(ctx, CTTS_GPU_ERR_BOUNDS, "output slot of utterance %u is misaligned, outside the buffer or smaller than its bound %llu",
                             s->utts + u, (unsigned long long)p->bounds[u]));
    if ((rc = grow_lane(s, l, p, packed)) != 0) return bail(rc);
    int16_t* const d_final = p->rs ? l.d_rs : l.d_out;   // the slots callers see
    p->d_out_last = d_final;
    cudaError_t e = cudaSuccess;
    if (n) {
        Launch launch{ctx, ctx->stream};
        rc = begin_run(ctx, p);
        if (!rc) rc = build_tasks(ctx, p, piece, ctx->stream);
        const auto tp2 = std::chrono::steady_clock::now();
        if (!rc) rc = launch_chain(launch, p, l.d_out, d_final);
        if (rc) return bail(rc);
        if (ctx->knobs.trace) {
            auto msf = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
            fprintf(stderr, "  submit %u utterances at %.1f ms: waited %.2f, prepare %.2f, build %.2f, launch %.2f ms\n", n, msf(s->t0, tp0),
                    msf(tsub0, tp0), msf(tp0, tp1), msf(tp1, tp2), msf(tp2, std::chrono::steady_clock::now()));
        }
        if (packed && (rc = encode_packed(launch, s, l, p, d_final)) != 0) return bail(rc);
        e = cudaEventRecord(l.kernels_done, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, l.kernels_done, 0);
        if (e == cudaSuccess && !packed) e = copy_slots(s, l, p, d_final, slot_off, slot_cap);
    } else {
        e = cudaEventRecord(l.copied, ctx->copy_stream);
    }
    if (e != cudaSuccess) return bail(fail(ctx, CTTS_GPU_ERR_CUDA, "enqueue: %s", cudaGetErrorString(e)));
    l.copy_pending = packed && n;   // packed mode: the copy is enqueued once the counts are on the host
    l.plan = p;
    l.user_counts = out_counts;
    l.user_offsets = offsets_out;
    l.user_bytes = out_bytes;
    l.utt_base = s->utts;
    l.n = n;
    l.busy = true;
    s->submitted++;
    s->utts += n;
    // packed mode: enqueue the copies of the pieces whose counts have arrived (in order; never blocks)
    pump_copies(s, 0);
    // hand over whatever has arrived in the meantime (never blocks)
    while (s->harvested < s->submitted) {
        ctts_gpu_ctx::Lane& h = ctx->lane[s->harvested % ctts_gpu_ctx::kLanes];
        if (h.busy && (h.copy_pending || cudaEventQuery(h.copied) != cudaSuccess)) break;
        harvest_one(s);
    }
    return s->error;
}

// Utterances u0 .. u1 - 1 of the plan as a plan of their own (the ops stay where they are)
ctts_batch_plan sub_plan(const ctts_batch_plan* plan, uint32_t u0, uint32_t u1) {
    return {u1 - u0, plan->n_ops, plan->utt_op_begin + u0, plan->speed + u0, plan->ops};
}

// Caller-defined slots: utterance u goes to pcm_out[off[u] ..), cap[u] samples of room.  The batch is cut into
// pieces of about piece_samples samples of slot space: the device->host copy of one overlaps the kernels of the
// next and the host-side compilation of the one after.
int submit_slot_pieces(ctts_gpu_session* s, const ctts_batch_plan* plan, const uint64_t* off, const uint64_t* cap,
                       uint32_t* out_counts) {
    const uint32_t n = plan->n_utts;
    int rc = CTTS_GPU_OK;
    uint64_t acc = 0;
    for (uint32_t u0 = 0, u = 0; u < n && !rc; u++) {
        acc += cap[u];
        if (acc >= s->ctx->knobs.piece_samples || u + 1 == n) {
            const ctts_batch_plan piece = sub_plan(plan, u0, u + 1);
            rc = submit_piece(s, &piece, off + u0, cap + u0, nullptr, out_counts + u0);
            u0 = u + 1;
            acc = 0;
        }
    }
    return rc;
}

int session_open(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, SessionOutput kind, void* out, uint64_t capacity,
                 ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** s_out) {
    if (!ctx || !params || !s_out || (capacity && !out)) return CTTS_GPU_ERR_INVALID_ARG;
    *s_out = nullptr;
    if (ctx->session) return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "a session is already open on this context");
    CU(ctx, cudaSetDevice(ctx->device));
    if (!ctx->copy_stream) CU(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (ctts_gpu_ctx::Lane& l : ctx->lane)
        for (cudaEvent_t* ev : {&l.kernels_done, &l.counts_ready, &l.copied})
            if (!*ev) CU(ctx, cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
    ctx->session = new ctts_gpu_session{ctx, *params, kind, static_cast<uint8_t*>(out), capacity, on_piece, user, std::chrono::steady_clock::now()};
    *s_out = ctx->session;
    return CTTS_GPU_OK;
}

// kind: the submit call's (either law for G.711)
int session_submit(ctts_gpu_session* s, SessionOutput kind, const ctts_batch_plan* piece, uint64_t* out_offsets,
                   uint32_t* out_bytes, uint32_t* out_counts) {
    const OutputKind& k = kOutput[s->kind];
    if (strcmp(k.submit, kOutput[kind].submit) != 0) return fail(s->ctx, CTTS_GPU_ERR_INVALID_ARG, "a %s session takes %s", k.name, k.submit);
    if (s->error) return s->error;
    CU(s->ctx, cudaSetDevice(s->ctx->device));
    return submit_piece(s, piece, nullptr, nullptr, out_offsets, out_counts, out_bytes);
}

}  // namespace

extern "C" {

int ctts_gpu_session_begin(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, int16_t* pcm_out, uint64_t capacity,
                           ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** out) {
    return session_open(ctx, params, OUT_PCM, pcm_out, capacity, on_piece, user, out);
}

int ctts_gpu_session_submit(ctts_gpu_session* s, const ctts_batch_plan* piece, uint64_t* out_offsets, uint32_t* out_counts) {
    if (!s || !piece || !out_counts || (piece->n_utts && !out_offsets)) return CTTS_GPU_ERR_INVALID_ARG;
    return session_submit(s, OUT_PCM, piece, out_offsets, nullptr, out_counts);
}

uint64_t ctts_gpu_flac_bound(uint64_t samples) {
    return ctts::FLAC_HEADER_BYTES + (samples + ctts::FLAC_BLOCK - 1) / ctts::FLAC_BLOCK * ctts::FLAC_FRAME_MAX;
}

int ctts_gpu_session_begin_flac(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, uint8_t* out, uint64_t capacity_bytes,
                                ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** s) {
    return session_open(ctx, params, OUT_FLAC, out, capacity_bytes, on_piece, user, s);
}

int ctts_gpu_session_submit_flac(ctts_gpu_session* s, const ctts_batch_plan* piece, uint64_t* out_offsets, uint32_t* out_bytes,
                                 uint32_t* out_counts) {
    if (!s || !piece || (piece->n_utts && (!out_offsets || !out_bytes || !out_counts))) return CTTS_GPU_ERR_INVALID_ARG;
    return session_submit(s, OUT_FLAC, piece, out_offsets, out_bytes, out_counts);
}

int ctts_gpu_session_begin_g711(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, int law, uint8_t* out,
                                uint64_t capacity_bytes, ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** s) {
    if (!ctx || !s || (capacity_bytes && !out)) return CTTS_GPU_ERR_INVALID_ARG;
    if (law != CTTS_GPU_G711_ULAW && law != CTTS_GPU_G711_ALAW) {
        *s = nullptr;
        return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "G.711 law %d: CTTS_GPU_G711_ULAW or CTTS_GPU_G711_ALAW", law);
    }
    return session_open(ctx, params, static_cast<SessionOutput>(law), out, capacity_bytes, on_piece, user, s);
}

int ctts_gpu_session_submit_g711(ctts_gpu_session* s, const ctts_batch_plan* piece, uint64_t* out_offsets, uint32_t* out_counts) {
    if (!s || !piece || !out_counts || (piece->n_utts && !out_offsets)) return CTTS_GPU_ERR_INVALID_ARG;
    return session_submit(s, OUT_ULAW, piece, out_offsets, nullptr, out_counts);
}

int ctts_gpu_session_end(ctts_gpu_session* s, uint64_t* samples_used) {
    if (!s) return CTTS_GPU_ERR_INVALID_ARG;
    ctts_gpu_ctx* ctx = s->ctx;
    cudaSetDevice(ctx->device);
    while (s->harvested < s->submitted) harvest_one(s);
    if (samples_used) *samples_used = s->cursor;
    if (ctx->knobs.trace)
        fprintf(stderr, "ctts_gpu session: %u utterances in %u pieces, %.1f MB to the host, %.1f ms\n", s->utts, s->submitted,
                1e-6 * (double)s->d2h_bytes, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - s->t0).count());
    const int rc = s->error;
    ctx->session = nullptr;
    delete s;
    return rc;
}

int ctts_gpu_synth_batch(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, const ctts_assembly_params* params,
                         int16_t* pcm_out, const uint64_t* out_offsets, uint32_t* out_counts) {
    return ctts_gpu_synth_batch_stream(ctx, plan, params, pcm_out, out_offsets, out_counts, nullptr, nullptr);
}

int ctts_gpu_synth_batch_stream(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, const ctts_assembly_params* params,
                                int16_t* pcm_out, const uint64_t* out_offsets, uint32_t* out_counts,
                                ctts_gpu_chunk_fn on_chunk, void* user) {
    if (!ctx || !plan || !params || !pcm_out || !out_offsets || !out_counts) return CTTS_GPU_ERR_INVALID_ARG;
    if (plan->n_utts && (!plan->utt_op_begin || !plan->speed)) return CTTS_GPU_ERR_INVALID_ARG;
    const uint32_t n = plan->n_utts;
    for (uint32_t u = 0; u < n; u++)
        if (out_offsets[u + 1] < out_offsets[u] || plan->utt_op_begin[u + 1] < plan->utt_op_begin[u] || plan->utt_op_begin[u + 1] > plan->n_ops)
            return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "offsets of utterance %u are not ascending", u);
    ctts_gpu_session* s = nullptr;
    int rc = ctts_gpu_session_begin(ctx, params, pcm_out, n ? out_offsets[n] : 0, on_chunk, user, &s);
    if (rc) return rc;
    std::vector<uint64_t> cap(std::max<uint32_t>(n, 1));
    for (uint32_t u = 0; u < n; u++) cap[u] = out_offsets[u + 1] - out_offsets[u];
    rc = submit_slot_pieces(s, plan, out_offsets, cap.data(), out_counts);
    const int rc_end = ctts_gpu_session_end(s, nullptr);
    return rc ? rc : rc_end;
}


// The same batch call with the library choosing the layout: packed output (exactly the samples that exist
// cross PCIe), offsets returned.  A session over the pieces of the plan.
int ctts_gpu_synth_batch_packed(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, const ctts_assembly_params* params,
                                int16_t* pcm_out, uint64_t capacity, uint64_t* out_offsets, uint32_t* out_counts,
                                uint64_t* samples_used) {
    if (!ctx || !plan || !params || !out_offsets || !out_counts || (capacity && !pcm_out)) return CTTS_GPU_ERR_INVALID_ARG;
    if (plan->n_utts && (!plan->utt_op_begin || !plan->speed)) return CTTS_GPU_ERR_INVALID_ARG;
    const uint32_t n = plan->n_utts;
    for (uint32_t u = 0; u < n; u++)
        if (plan->utt_op_begin[u + 1] < plan->utt_op_begin[u] || plan->utt_op_begin[u + 1] > plan->n_ops)
            return fail(ctx, CTTS_GPU_ERR_INVALID_ARG, "ops of utterance %u are not ascending", u);
    ctts_gpu_session* s = nullptr;
    int rc = ctts_gpu_session_begin(ctx, params, pcm_out, capacity, nullptr, nullptr, &s);
    if (rc) return rc;
    // pieces of about piece_samples / 2400 utterances ... by ops: an op appends at most a few thousand samples, so
    // cut by op count (no bounds are known before a piece is compiled): ~70 k ops ~ 192 sentences of 200 characters (measured: text -> PCM of a mixed-speed batch 105 ms with pieces of
    // 128, 97 with 192, 99 with 256; at speed 1.0 no difference)
    const uint64_t ops_per_piece = std::max<uint64_t>(ctx->knobs.piece_samples / 2800, 64);
    for (uint32_t u0 = 0, u = 0; u < n && !rc; u++) {
        if (plan->utt_op_begin[u + 1] - plan->utt_op_begin[u0] >= ops_per_piece || u + 1 == n) {
            const ctts_batch_plan piece = sub_plan(plan, u0, u + 1);
            rc = submit_piece(s, &piece, nullptr, nullptr, out_offsets + u0, out_counts + u0);
            u0 = u + 1;
        }
    }
    const int rc_end = ctts_gpu_session_end(s, samples_used);
    return rc ? rc : rc_end;
}

// ---------------------------------------------------------------- one batch on several GPUs

// Utterances are independent (no state crosses ctts_synthesize calls, ctts.c:3623, except the read-only
// voice): the batch is partitioned by utterance -- greedy longest-processing-time on the host-known slot
// sizes, every device holding its own replica of the voice (one context each) -- and every shard is run
// by its own host thread as a session that delivers straight into the caller's buffer at the
// utterance's own slot: the host gather is the layout itself, there is no data-path collective.
int ctts_gpu_multi_synth_batch(ctts_gpu_ctx* const* ctxs, uint32_t n_ctx, const ctts_batch_plan* plan,
                               const ctts_assembly_params* params, int16_t* pcm_out, const uint64_t* out_offsets,
                               uint32_t* out_counts, uint32_t* shard_of) {
    if (!ctxs || !n_ctx || !plan || !params || !pcm_out || !out_offsets || !out_counts) return CTTS_GPU_ERR_INVALID_ARG;
    for (uint32_t d = 0; d < n_ctx; d++)
        if (!ctxs[d]) return CTTS_GPU_ERR_INVALID_ARG;
    for (uint32_t d = 1; d < n_ctx; d++)
        if ((ctxs[d]->rs ? ctxs[d]->rs->hz : CTTS_PLAN_SAMPLE_RATE) != (ctxs[0]->rs ? ctxs[0]->rs->hz : CTTS_PLAN_SAMPLE_RATE))
            return fail(ctxs[0], CTTS_GPU_ERR_INVALID_ARG, "context %u has another output rate than context 0", d);
    for (uint32_t d = 1; d < n_ctx; d++) {
        const ctts_gpu_ctx::LdTable *a = ctxs[d]->ld, *b = ctxs[0]->ld;
        if ((a == nullptr) != (b == nullptr) || (a && (a->target != b->target || a->ceiling != b->ceiling || a->true_peak != b->true_peak)))
            return fail(ctxs[0], CTTS_GPU_ERR_INVALID_ARG, "context %u has another loudness setting than context 0", d);
    }
    if (plan->n_utts && (!plan->utt_op_begin || !plan->speed)) return CTTS_GPU_ERR_INVALID_ARG;
    const uint32_t n = plan->n_utts;
    for (uint32_t u = 0; u < n; u++)
        if (out_offsets[u + 1] < out_offsets[u] || plan->utt_op_begin[u + 1] < plan->utt_op_begin[u] || plan->utt_op_begin[u + 1] > plan->n_ops)
            return fail(ctxs[0], CTTS_GPU_ERR_INVALID_ARG, "offsets of utterance %u are not ascending", u);
    // ---- LPT partition; the cost of an utterance is its slot size (what has to cross PCIe), plus its
    //      pre-stretch length when it goes through WSOLA
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    std::vector<uint64_t> cost(n);
    for (uint32_t u = 0; u < n; u++) {
        cost[u] = out_offsets[u + 1] - out_offsets[u];
        uint32_t hop = 0;
        if (needs_stretch(plan->speed[u], &hop)) cost[u] += (cost[u] * 128) / std::max<uint32_t>(hop, 1);
    }
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return cost[a] > cost[b]; });
    std::vector<std::vector<uint32_t>> shard(n_ctx);
    {
        std::vector<uint64_t> load(n_ctx, 0);
        for (const uint32_t u : order) {
            const uint32_t d = (uint32_t)(std::min_element(load.begin(), load.end()) - load.begin());
            shard[d].push_back(u);
            load[d] += cost[u];
        }
        for (std::vector<uint32_t>& sh : shard) std::sort(sh.begin(), sh.end());   // batch order inside a shard
    }
    if (shard_of)
        for (uint32_t d = 0; d < n_ctx; d++)
            for (const uint32_t u : shard[d]) shard_of[u] = d;

    // ---- one host thread per device
    std::vector<int> rcs(n_ctx, 0);
    auto run_shard = [&](uint32_t d) {
        ctts_gpu_ctx* ctx = ctxs[d];
        const std::vector<uint32_t>& mine = shard[d];
        const uint32_t m = (uint32_t)mine.size();
        if (!m) return;
        // the shard as a plan of its own (CSR needs contiguous ops) and the slots of its utterances
        std::vector<uint32_t> begin((size_t)m + 1, 0);
        std::vector<float> speed(m);
        std::vector<uint64_t> off(m), cap(m);
        std::vector<uint32_t> counts(m, 0);
        uint64_t n_ops = 0;
        for (uint32_t i = 0; i < m; i++) n_ops += plan->utt_op_begin[mine[i] + 1] - plan->utt_op_begin[mine[i]];
        if (n_ops > 0xffffffffull) { rcs[d] = CTTS_GPU_ERR_INVALID_ARG; return; }
        std::vector<ctts_plan_op> ops((size_t)std::max<uint64_t>(n_ops, 1));
        uint32_t at = 0;
        for (uint32_t i = 0; i < m; i++) {
            const uint32_t u = mine[i], b = plan->utt_op_begin[u], e = plan->utt_op_begin[u + 1];
            if (e > b) memcpy(ops.data() + at, plan->ops + b, (size_t)(e - b) * sizeof(ctts_plan_op));
            at += e - b;
            begin[i + 1] = at;
            speed[i] = plan->speed[u];
            off[i] = out_offsets[u];
            cap[i] = out_offsets[u + 1] - out_offsets[u];
        }
        ctts_batch_plan sub{m, (uint32_t)n_ops, begin.data(), speed.data(), ops.data()};
        ctts_gpu_session* s = nullptr;
        int rc = ctts_gpu_session_begin(ctx, params, pcm_out, out_offsets[n], nullptr, nullptr, &s);
        if (rc) { rcs[d] = rc; return; }
        rc = submit_slot_pieces(s, &sub, off.data(), cap.data(), counts.data());
        const int rc_end = ctts_gpu_session_end(s, nullptr);
        rcs[d] = rc ? rc : rc_end;
        for (uint32_t i = 0; i < m; i++) out_counts[mine[i]] = counts[i];
    };
    std::vector<std::thread> th;
    for (uint32_t d = 1; d < n_ctx; d++) th.emplace_back(run_shard, d);
    run_shard(0);
    for (std::thread& t : th) t.join();
    for (uint32_t d = 0; d < n_ctx; d++)
        if (rcs[d]) {
            if (d) snprintf(ctxs[0]->err, sizeof ctxs[0]->err, "device %u: %.480s", d, ctxs[d]->err);
            return rcs[d];
        }
    return CTTS_GPU_OK;
}

}  // extern "C"
