/*
 * ctts_gpu.h -- C-ABI of the B200 (sm_100a) batched audio-assembly back end.
 *
 * Exported by libctts_gpu.so.  Plain pointers and sizes only.  This is the
 * boundary the reference does not have: it replaces every sample-touching
 * statement of `ctts_synthesize` (ctts.c:3689-3921) -- unit gather
 * (get_unit_samples :1557), normalize_rms :1709, smooth_pitch_boundary :1979,
 * match_boundary_energy :1730, buffer_append_crossfade :3279,
 * buffer_append_silence :3361, apply_fade_out :3028, remove_silence_regions
 * :1634, apply_phrase_intonation :2736, time_stretch :3490 -- for a whole batch
 * of utterances described by a CSR plan (ctts_plan.h) that the unchanged host
 * front end emits.
 *
 * Conventions follow the reference API (ctts.h:175-346): 0 on success,
 * negative CTTS_ERR_* on failure (plus CTTS_GPU_ERR_* below); caller-owned
 * output buffers (no hidden malloc per utterance); one context per GPU; a
 * context is used by one host thread at a time.  There is NO CPU fallback:
 * without a CUDA device every entry point fails with CTTS_GPU_ERR_CUDA.
 */
#ifndef CTTS_GPU_H
#define CTTS_GPU_H

#include "ctts_plan.h"

#ifdef __cplusplus
extern "C" {
#endif

#define CTTS_GPU_OK 0
#define CTTS_GPU_ERR_INVALID_ARG (-1)    /* == CTTS_ERR_INVALID_ARG */
#define CTTS_GPU_ERR_INVALID_FORMAT (-5) /* == CTTS_ERR_INVALID_FORMAT (voice.db) */
#define CTTS_GPU_ERR_OUT_OF_MEMORY (-6)  /* == CTTS_ERR_OUT_OF_MEMORY */
#define CTTS_GPU_ERR_VERSION (-8)        /* == CTTS_ERR_VERSION */
#define CTTS_GPU_ERR_CUDA (-100)         /* CUDA runtime error, see ctts_gpu_last_error */
#define CTTS_GPU_ERR_BOUNDS (-101)       /* an output slot is smaller than its upper bound */
#define CTTS_GPU_ERR_DEVICE (-102)       /* a kernel reported an internal capacity error */

typedef struct ctts_gpu_ctx ctts_gpu_ctx;
typedef struct ctts_gpu_plan ctts_gpu_plan;

/* Replaces ctts_init (ctts.c:1117) for the back end: parses the same voice.db
 * bytes (header ctts.h:84-98, index :101-111), re-packs the PCM pool so every
 * unit starts 16-byte aligned, uploads it with the fade LUTs (ctts.c:60-73)
 * and Hann windows (ctts.c:1624, :2198), all computed on the host with libm. */
int ctts_gpu_init(ctts_gpu_ctx** out, const void* voice_db, size_t db_size, int device_ordinal);
/* Replaces ctts_free (ctts.c:1167). */
void ctts_gpu_free(ctts_gpu_ctx* ctx);
/* Kernels and copies are issued on `cuda_stream` (a cudaStream_t); NULL
 * restores the context's own stream. */
int ctts_gpu_set_stream(ctts_gpu_ctx* ctx, void* cuda_stream);
/* Output sample rate of the context (DESIGN.md 3.4).  The back end assembles at the native 22 050 Hz
 * (CTTS_PLAN_SAMPLE_RATE); any other rate converts every utterance on the device, after time stretching and
 * before it is packed or copied: a Kaiser-windowed sinc of 2*40*max(L, M) + 1 taps at the reduced ratio L/M =
 * hz/22050, utterance n samples long -> ceil(n*L/M) samples.  Accepted: integer hz in [8000, 48000] with
 * max(L, M) <= 1024 (8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000 among them).  Builds and uploads the
 * tap table (once per rate and context).  CTTS_GPU_ERR_INVALID_ARG for any other rate and while a session is
 * open; the context is then unchanged.  22050 (the default) enqueues no conversion at all.
 *
 * EVERY count, offset, capacity and bound of the context is in output-rate samples: ctts_gpu_plan_bounds, all
 * ctts_gpu_synth_batch* calls, sessions, resident plans (out_samples, out_offsets, read_counts, read_pcm; a plan
 * keeps the rate it was created under) and ctts_gpu_multi_synth_batch, which rejects contexts whose rates
 * differ.  ctts_gpu_plan_read_pre stays at the native rate. */
int ctts_gpu_set_output_rate(ctts_gpu_ctx* ctx, uint32_t hz);
/* Loudness normalization of the context (DESIGN.md 3.6), off by default.  Every utterance's integrated loudness L is
 * measured after ITU-R BS.1770-4 on its output-rate samples x (K-weighting in double, 400 ms blocks, absolute gate
 * -70 LUFS, relative gate -10 LU; L is undefined for utterances shorter than 400 ms or with no block above the gates),
 * and one gain per utterance is applied on the device, after the rate conversion and before the output is packed,
 * encoded or copied:
 *   k = clamp(floor(100 * (T - L) + 0.5), -8000, 8000), G = min(floor(65536 * 10^(k / 2000)), floor(A * 65536 / P))
 *   with A = floor(32767 * 10^(C / 20)) and P = max |x|; G = 65536 when L is undefined;  y = (x * G + 32768) >> 16.
 * So an utterance reaches T LUFS to 0.005 LU unless its SAMPLE peak would pass C dBFS (no compression; for a
 * true-peak ceiling see ctts_gpu_set_loudness_true_peak); G = 65536 leaves it exactly as it was; counts do not change.
 * Accepted: target_lufs a finite T in [-60, -5] with ceiling_dbfs a finite C in [-20, 0]; target_lufs == 0 turns the
 * stage off (then nothing is enqueued: bytes and kernel launches are those of a context that never set it).
 * Builds the K-weighting of the context's output rate (and keeps it consistent when the rate changes) and, once per
 * context, uploads the gain table.  CTTS_GPU_ERR_INVALID_ARG for anything else and while a session is open; the context
 * is then unchanged.
 *
 * It applies to every path: resident plans (a plan keeps the setting it was created under), all ctts_gpu_synth_batch*
 * calls, PCM, FLAC and G.711 sessions, ctts_b200_synth_texts(_flac, _g711) and ctts_gpu_multi_synth_batch, which
 * rejects contexts whose settings differ. */
int ctts_gpu_set_loudness(ctts_gpu_ctx* ctx, float target_lufs, float ceiling_dbfs);
/* The same loudness normalization with a TRUE-PEAK ceiling of C dBTP (ITU-R BS.1770-4 Annex 2, DESIGN.md 3.6), for
 * delivery specifications such as EBU R128 (-1 dBTP).  The peak is that of the signal interpolated 4x with the 49-tap
 * windowed sinc h[j] = sinc((j - 24) / 4) * 0.5 * (1 - cos(2 pi j / 48)), j = 0 .. 48 (|h[j]| <= 1e-9 set to 0, taps
 * rounded to float once), the utterance taken as zero outside its n samples:
 *   v[m] = sum over j of x[j] * h[m - 4j + 24] for m = -24 .. 4(n - 1) + 24 (ascending j, one fmaf per term from 0.0f),
 *   P = max |v[m]| (>= max |x|, since v[4j] = x[j]),  G = min(floor(65536 * 10^(k / 2000)), floor((A - 1) * 65536 / P))
 *   (the division in double), everything else as ctts_gpu_set_loudness.
 * Guarantee: the interpolated peak of the delivered y (same taps, exact arithmetic) is <= A, so |y| <= A.
 * The same acceptance rules; it replaces the context's loudness setting, whichever kind that was, and
 * ctts_gpu_set_loudness replaces it back.  Plans keep the kind, it follows the output rate, and
 * ctts_gpu_multi_synth_batch rejects contexts whose kinds differ.  A plan adds ceil(n / 65535) kernel launches. */
int ctts_gpu_set_loudness_true_peak(ctts_gpu_ctx* ctx, float target_lufs, float ceiling_dbtp);
/* Text of the last error of a context; ctx == NULL: why the calling thread's last ctts_gpu_init failed. */
const char* ctts_gpu_last_error(const ctts_gpu_ctx* ctx);

/* Upper bound, per utterance, of the samples ctts_gpu_synth_batch may write
 * (sum of unit lengths and silences; for speed != 1.0f the WSOLA bound
 * num_frames*synthesis_hop + 512 of ctts.c:3515-3517). */
int ctts_gpu_plan_bounds(const ctts_gpu_ctx* ctx, const ctts_batch_plan* plan, uint64_t* out_bound);

/* THE drop-in entry point: replaces the sample half of N calls of
 * ctts_synthesize (ctts.c:3623).  Host buffers in, host buffers out,
 * synchronous on return.  Utterance u's PCM is written to
 * pcm_out[out_offsets[u] .. out_offsets[u] + out_counts[u]); out_offsets has
 * n_utts+1 entries, each a multiple of 8 samples, and
 * out_offsets[u+1]-out_offsets[u] must be >= ctts_gpu_plan_bounds()[u].  Samples of a slot past
 * out_counts[u] are unspecified (they may hold PCM of an earlier call on this context). */
int ctts_gpu_synth_batch(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan,
                         const ctts_assembly_params* params, int16_t* pcm_out,
                         const uint64_t* out_offsets, uint32_t* out_counts);

/* The same call with the library choosing the layout: the output is PACKED -- a device prefix sum of the counts
 * places every utterance right behind the one before it (rounded up to 8 samples; the padding is zero), a device
 * gather moves the samples there, and exactly those samples cross PCIe (a slot sized by a bound carries whatever
 * silence trimming removed, 4.9 % on the benchmark corpus).  out_offsets (n_utts entries, written by the call) says
 * where each utterance landed; capacity: ctts_gpu_plan_bounds summed (rounded up to 8 each) is always enough, less
 * fails with CTTS_GPU_ERR_BOUNDS; *samples_used (may be NULL) is the space taken. */
int ctts_gpu_synth_batch_packed(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan,
                                const ctts_assembly_params* params, int16_t* pcm_out, uint64_t capacity,
                                uint64_t* out_offsets, uint32_t* out_counts, uint64_t* samples_used);

/* The same call, streaming: `on_chunk(user, utt_begin, utt_end)` is invoked on the calling thread, in
 * utterance order, as soon as the PCM and the counts of utterances [utt_begin, utt_end) are in host
 * memory -- while the device is still working on later utterances -- so the caller can write WAV files
 * (ctts_write_wav, ctts.c:809) or hand audio on without waiting for the batch (the output path of a
 * 65 536-paragraph batch is 87 GB of PCM, SURVEY.md 8f).  A range that holds an utterance with a device-side
 * error is not handed over, nor is any range after it; the error is the return value.
 * on_chunk == NULL: ctts_gpu_synth_batch. */
typedef void (*ctts_gpu_chunk_fn)(void* user, uint32_t utt_begin, uint32_t utt_end);
int ctts_gpu_synth_batch_stream(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan,
                                const ctts_assembly_params* params, int16_t* pcm_out,
                                const uint64_t* out_offsets, uint32_t* out_counts,
                                ctts_gpu_chunk_fn on_chunk, void* user);

/* ---- sessions: ONE batch fed in pieces --------------------------------------------------------------
 * The reference interleaves text work and sample work inside one call (ctts.c:3638-3655, :3689-3871).  A
 * session gives the batch equivalent: the caller plans piece c+1 (the text front end, on host threads)
 * while the device assembles piece c and piece c-1 travels to pcm_out.  ctts_gpu_synth_batch(_stream) is a
 * session over the pieces of one plan; ctts_b200_synth_texts (ctts_b200.h) is a session fed by the front end.
 *
 * begin    pcm_out (page-locked for full copy speed) holds `capacity` samples; on_piece (may be NULL) is called
 *          on the submitting thread, in order, with the session-wide utterance range of every piece whose PCM
 *          and counts have arrived.
 * submit   asynchronous: returns as soon as the piece is compiled and enqueued (up to four pieces are in
 *          flight; a fifth waits for the oldest).  The output is PACKED: a device prefix sum of the counts
 *          places every utterance right behind the one before it (rounded up to 8 samples, so every utterance
 *          starts 16-byte aligned; the padding is zero), a device gather moves the samples there, and exactly
 *          those samples cross PCIe.  out_offsets[i] and out_counts[i] (n entries each) are written when the
 *          piece has arrived -- before on_piece is called for it, at the latest by ctts_gpu_session_end; the
 *          plan may be freed when submit returns.  A buffer that turns out too small ends the session with
 *          CTTS_GPU_ERR_BOUNDS (ctts_gpu_plan_bounds gives what is always enough).
 * end      waits for everything, returns the first error of the session; *samples_used (may be NULL) is
 *          the space taken in pcm_out.
 * One session per context at a time. */
typedef struct ctts_gpu_session ctts_gpu_session;
int ctts_gpu_session_begin(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, int16_t* pcm_out,
                           uint64_t capacity, ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** out);
int ctts_gpu_session_submit(ctts_gpu_session* s, const ctts_batch_plan* piece, uint64_t* out_offsets,
                            uint32_t* out_counts);
int ctts_gpu_session_end(ctts_gpu_session* s, uint64_t* samples_used);

/* ---- FLAC sessions: the same session, every utterance delivered as one .flac file (DESIGN.md 3.5) ----------------
 * Lossless: a file decodes to exactly the PCM a PCM session delivers for the same piece.  Each file is complete and
 * self-contained (RFC 9639): "fLaC", one STREAMINFO block (the context's output rate, mono, 16 bit, the utterance's
 * sample count, MD5 all zero), frames of 4096 samples (the last one holds the remainder) with CONSTANT, FIXED
 * (orders 0-4, Rice-coded residuals) or VERBATIM subframes.  The encoder is deterministic.
 * begin_flac   as ctts_gpu_session_begin; out (page-locked for full copy speed) holds capacity_bytes bytes.
 * submit_flac  as ctts_gpu_session_submit; the files are packed back to back in out, each starting at a multiple of
 *              16 bytes (the padding is zero).  out_offsets[i] (bytes), out_bytes[i] (file size) and out_counts[i]
 *              (samples) are written when the piece has arrived.  A buffer that turns out too small ends the session
 *              with CTTS_GPU_ERR_BOUNDS; ctts_gpu_flac_bound of every bound (rounded up to 16) is always enough.
 * ctts_gpu_session_end closes it; *samples_used is then the number of BYTES taken in out.  ctts_gpu_session_submit on
 * a FLAC session, or ctts_gpu_session_submit_flac on a PCM session, is CTTS_GPU_ERR_INVALID_ARG. */
int ctts_gpu_session_begin_flac(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, uint8_t* out,
                                uint64_t capacity_bytes, ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** s);
int ctts_gpu_session_submit_flac(ctts_gpu_session* s, const ctts_batch_plan* piece, uint64_t* out_offsets,
                                 uint32_t* out_bytes, uint32_t* out_counts);
/* Largest .flac file of an utterance of `samples` samples: 42 + ceil(samples / 4096) * (16 + 1 + 8192 + 2) bytes
 * (a VERBATIM subframe caps every frame). */
uint64_t ctts_gpu_flac_bound(uint64_t samples);

/* ---- G.711 sessions: the same session, every sample delivered as one μ-law or A-law byte (DESIGN.md 3.7) --------
 * For telephony: 8-bit G.711 at the context's output rate (8000 Hz for the classic telephone channel), as IVR and
 * contact-center systems play it.  The encoder is the ITU-T G.711 reference (the G.191 tools, Sun's g711.c, CPython's
 * audioop.lin2ulaw / lin2alaw on 16-bit input), applied to the int16 samples a PCM session delivers for the same piece
 * on the same context settings (after assembly, time stretching, rate conversion and loudness):
 *   μ-law  v = x >> 2 (arithmetic); m = min(|v|, 8159) + 33; segment s = the first of 0..7 with m <= (64 << s) - 1
 *          (none: code 0x7F), else code = (s << 4) | ((m >> (s + 1)) & 0xF); the byte is code ^ 0x7F for v < 0,
 *          code ^ 0xFF otherwise.
 *   A-law  v = x >> 3; m = -v - 1 for v < 0, else v; s = the first of 0..7 with m <= (32 << s) - 1;
 *          code = (s << 4) | ((m >> max(s, 1)) & 0xF); the byte is code ^ 0x55 for v < 0, code ^ 0xD5 otherwise.
 * No zero-code suppression.  E.g. x = 0, -1, 100, -100, 32767, -32768 -> μ-law ff 7e f2 72 80 00, A-law d5 55 d3 53 aa 2a.
 * Layout: the PCM session's packed layout with bytes in place of samples.  Utterance u is out[out_offsets[u] ..
 * out_offsets[u] + out_counts[u]), one byte per sample; every offset is a multiple of 8 and the next utterance starts
 * at out_offsets[u] + up8(out_counts[u]); the padding bytes hold the law's code for silence (0xFF μ-law, 0xD5 A-law),
 * not zero (a zero byte decodes to a near full-scale sample).
 * begin_g711   as ctts_gpu_session_begin with law CTTS_GPU_G711_ULAW or CTTS_GPU_G711_ALAW; out (page-locked for full
 *              copy speed) holds capacity_bytes bytes.  The sum of up8(bound) over the ctts_gpu_plan_bounds, read as
 *              bytes, is always enough.
 * submit_g711  as ctts_gpu_session_submit, offsets in bytes.  A buffer that turns out too small ends the session with
 *              CTTS_GPU_ERR_BOUNDS.
 * ctts_gpu_session_end closes it; *samples_used is then the number of BYTES taken in out.  Any other law, a second
 * session on the context, and a submit call of another kind on a G.711 session (or submit_g711 on a PCM or FLAC
 * session) is CTTS_GPU_ERR_INVALID_ARG. */
#define CTTS_GPU_G711_ULAW 1
#define CTTS_GPU_G711_ALAW 2
int ctts_gpu_session_begin_g711(ctts_gpu_ctx* ctx, const ctts_assembly_params* params, int law, uint8_t* out,
                                uint64_t capacity_bytes, ctts_gpu_chunk_fn on_piece, void* user, ctts_gpu_session** s);
int ctts_gpu_session_submit_g711(ctts_gpu_session* s, const ctts_batch_plan* piece, uint64_t* out_offsets,
                                 uint32_t* out_counts);

/* ---- one batch on several GPUs of one box ---------------------------------------------------------
 * ctxs[d] is a context on device d (each holds its own replica of the voice: ctts_gpu_init per device).
 * The batch is partitioned by utterance (greedy longest-processing-time on the slot sizes, WSOLA
 * utterances weighted up), every shard runs on its own host thread and device and delivers straight into
 * the caller's buffer at the utterance's slot: the host-side gather of BASELINE's multi-GPU configuration,
 * no data-path collective.  Arguments as ctts_gpu_synth_batch; shard_of (may be NULL, n_utts entries)
 * receives the device every utterance ran on.  The contexts must not be in use by other threads. */
int ctts_gpu_multi_synth_batch(ctts_gpu_ctx* const* ctxs, uint32_t n_ctx, const ctts_batch_plan* plan,
                               const ctts_assembly_params* params, int16_t* pcm_out,
                               const uint64_t* out_offsets, uint32_t* out_counts, uint32_t* shard_of);

/* ---- resident-plan path: upload once, run many times, PCM stays in HBM ---- */

/* Uploads the plan, derives the region tasks and output layout
 * (slots sized by the bounds, 16-byte aligned) and allocates workspace.
 * `out_offsets` may be NULL (packed slots chosen by the library). */
int ctts_gpu_plan_create(ctts_gpu_ctx* ctx, const ctts_batch_plan* plan,
                         const ctts_assembly_params* params, const uint64_t* out_offsets,
                         ctts_gpu_plan** out);
void ctts_gpu_plan_destroy(ctts_gpu_plan* plan);
/* total samples spanned by the output slots, and the slot offsets (n_utts+1) */
uint64_t ctts_gpu_plan_out_samples(const ctts_gpu_plan* plan);
int ctts_gpu_plan_out_offsets(const ctts_gpu_plan* plan, uint64_t* offsets);
/* Enqueue the kernels for the whole batch on the context stream (asynchronous).
 * d_pcm_out: device buffer of >= ctts_gpu_plan_out_samples() int16, or NULL to
 * use a buffer owned by the plan. */
int ctts_gpu_plan_run(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, int16_t* d_pcm_out);
/* Waits for the stream, then copies counts (and checks device error flags). */
int ctts_gpu_plan_read_counts(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, uint32_t* out_counts);
/* Device -> host copy of the plan-owned PCM buffer range [first, first+n). */
int ctts_gpu_plan_read_pcm(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, int16_t* dst, uint64_t first,
                           uint64_t n);
/* After a run of a plan created with loudness normalization on: L (LUFS, -INFINITY when undefined) and G (Q16) of
 * every utterance, n_utts entries each.  CTTS_GPU_ERR_INVALID_ARG for a plan created with the stage off. */
int ctts_gpu_plan_read_loudness(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, double* lufs, uint32_t* gain);
/* After a run of a plan created under a true-peak setting (ctts_gpu_set_loudness_true_peak): every utterance's true
 * peak P before the gain (int16 units), n_utts entries.  CTTS_GPU_ERR_INVALID_ARG for any other plan. */
int ctts_gpu_plan_read_true_peak(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, float* peak);
/* Debug / tests: pre-stretch buffer of utterance u (only for speed != 1.0f utterances). */
int ctts_gpu_plan_read_pre(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, uint32_t u, int16_t* dst,
                           uint64_t cap, uint64_t* n);

/* After a run: how time_stretch's frame chain (ctts.c:3555-3592) was resolved.  The back end speculates
 * every frame's analysis offset (the previous frame's, or -128 behind digital silence), verifies all frames
 * independently, and walks the chain frame by frame only from an utterance's first unverified frame on. */
typedef struct ctts_gpu_wsola_stats {
    uint64_t frames;             /* WSOLA frames of the batch */
    uint64_t tier2_candidates;   /* candidates the partial-sum bound could not reject (full 384-term filter score) */
    uint64_t exact_evaluations;  /* ... of those, and of the chain walk's decisions: the reference's exact loop */
    uint64_t walked_utterances;  /* utterances with an unverified frame */
    uint64_t walked_frames;      /* frames decided by the chain walk */
} ctts_gpu_wsola_stats;
int ctts_gpu_plan_wsola_stats(ctts_gpu_ctx* ctx, ctts_gpu_plan* plan, ctts_gpu_wsola_stats* out);

typedef struct ctts_gpu_run_info {
    uint32_t kernel_launches;    /* kernels enqueued by one ctts_gpu_plan_run */
    uint32_t n_stretch;          /* utterances that go through WSOLA */
    uint64_t gather_samples;     /* sum of unit lengths over the batch (PCM pool reads) */
    uint64_t bound_samples;      /* sum of output upper bounds */
    uint32_t smem_bytes;         /* dynamic shared memory of the assembly kernel */
    uint32_t window_samples;     /* shared-memory window capacity per CTA */
    uint32_t halo_samples;       /* unit-head staging capacity per CTA */
    uint32_t threads;
    uint32_t n_tasks;            /* region tasks of the assembly kernel */
    uint32_t n_global_tasks;     /* of those: regions larger than the window, assembled in the HBM slot */
    uint32_t ctas_per_sm;        /* resident CTAs per SM of the assembly kernel */
    uint32_t grid;               /* persistent CTAs launched */
    /* word-region deduplication: equal word regions of a batch are assembled once per launch (canonical tasks),
     * every other occurrence copies the result and runs its own contour */
    uint32_t n_canon_tasks;      /* distinct regions computed once */
    uint32_t n_dedup_tasks;      /* region tasks that take their samples from one of those */
    uint64_t dedup_bound_samples;/* sum of their upper bounds */
    /* ... second level: tasks that are equal as a whole (same region, same contour factors, same pause behind it) */
    uint32_t n_source_tasks;     /* tasks whose samples are also kept for the others */
    uint32_t n_reuse_tasks;      /* tasks that copy them and run nothing */
    uint64_t reuse_bound_samples;/* sum of the upper bounds of those */
} ctts_gpu_run_info;
int ctts_gpu_plan_info(const ctts_gpu_plan* plan, ctts_gpu_run_info* info);

/* Page-locked host memory for the caller's PCM buffer (the device->host copies of
 * ctts_gpu_synth_batch run at PCIe speed into it; pageable memory works too, slower).  The
 * reference hands out malloc'ed sample buffers (ctts_synthesize / ctts_free_samples, ctts.h:212-224);
 * these are the batch equivalents for a plain-C host that does not link the CUDA runtime itself. */
void* ctts_gpu_host_alloc(size_t bytes);
void ctts_gpu_host_free(void* p);

#ifdef __cplusplus
}
#endif

#endif /* CTTS_GPU_H */
