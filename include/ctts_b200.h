/*
 * ctts_b200.h -- text in, PCM out: the whole `ctts synth` path (ctts_synthesize, ctts.c:3623) for a batch,
 * the text front end (ctts_front.h, host threads) pipelined into the B200 back end (ctts_gpu.h).
 *
 * Exported by libctts_b200.so (plain C over the two C-ABI libraries; what the `ctts_b200` command line and
 * a CTTS maintainer's batch driver link).  The reference does text work and sample work of one utterance
 * inside one call (ctts.c:3638-3655 normalisation, :3689-3871 the walk with unit selection :1406); here the
 * batch is cut into groups of 16 utterances, a pool of planner threads turns groups into plans
 * (ctts_front_plan_batch_threads) while the calling thread joins the plans that are ready, in order, into
 * pieces and feeds them to a ctts_gpu_session: planning of piece c+1 overlaps the kernels of piece c and the
 * device->host copy of piece c-1.  Plans are byte-identical to what ctts_front_plan_batch returns for the whole batch.
 */
#ifndef CTTS_B200_H
#define CTTS_B200_H

#include "ctts_front.h"
#include "ctts_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

/* A plan cache: the plan of an utterance depends on its text alone (for one front end handle: voice index, config,
 * rules; the speed travels beside the ops), so a caller that sees the same sentences again can skip the text half.
 * Entries are immutable and never evicted; the cache stops taking entries at max_bytes.  Thread safe.  Use one
 * cache per front end handle. */
typedef struct ctts_b200_plan_cache ctts_b200_plan_cache;
ctts_b200_plan_cache* ctts_b200_plan_cache_create(size_t max_bytes);
void ctts_b200_plan_cache_destroy(ctts_b200_plan_cache* cache);
void ctts_b200_plan_cache_stats(ctts_b200_plan_cache* cache, uint64_t* hits, uint64_t* misses, uint64_t* entries,
                                uint64_t* bytes);

typedef struct ctts_b200_options {
    uint32_t piece_utts;     /* most utterances per device piece (0: 192); planner jobs are groups of 16 */
    uint32_t threads;        /* planner threads (0: host cores - 1, at least 1, at most 32) */
    ctts_gpu_chunk_fn on_piece;   /* may be NULL: called in order as utterance ranges arrive in pcm_out */
    void* user;
    ctts_b200_plan_cache* cache;  /* may be NULL */
} ctts_b200_options;

/* Timing of one call, for bench.py and the command line (seconds since the call began). */
typedef struct ctts_b200_timing {
    double first_plan_s;     /* first piece planned */
    double all_plans_s;      /* last piece planned */
    double all_submitted_s;  /* last piece handed to the device */
    double done_s;           /* everything in pcm_out */
    double wait_for_plans_s; /* time the submitting thread spent waiting for the planners */
    uint32_t pieces;         /* pieces submitted to the device */
    uint32_t reserved;
} ctts_b200_timing;

/* N texts -> PCM at the output rate of `gpu` (ctts_gpu_set_output_rate; every count, offset and capacity is in
 * samples of that rate).  pcm_out (ctts_gpu_host_alloc) holds `capacity` samples; utterance u lands at
 * pcm_out[out_offsets[u] .. out_offsets[u] + out_counts[u]) (out_offsets: n entries; the utterances are
 * packed back to back, each starting 16-byte aligned; *samples_used, may be NULL, = space taken).  speeds may be NULL
 * (all 1.0); stats may be NULL (2n: units found, missing per utterance, ctts.c:3861, :3866).
 * Returns 0 or the first CTTS_FRONT_ERR_* / CTTS_GPU_ERR_* code.  CTTS_GPU_ERR_BOUNDS: capacity too small
 * (ctts_b200_capacity_hint gives a safe size). */
int ctts_b200_synth_texts(ctts_front* front, ctts_gpu_ctx* gpu, const char* const* texts, const float* speeds,
                          uint32_t n, int16_t* pcm_out, uint64_t capacity, uint64_t* out_offsets,
                          uint32_t* out_counts, uint32_t* stats, uint64_t* samples_used,
                          const ctts_b200_options* opt, ctts_b200_timing* timing);

/* A capacity (samples) that is enough for the texts: characters x the longest unit x the slowest speed,
 * without planning anything.  At another output rate: ctts_b200_capacity_hint_rate (ctts_b200_rate.h). */
uint64_t ctts_b200_capacity_hint(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n);

#ifdef __cplusplus
}
#endif

#include "ctts_b200_rate.h"
#include "ctts_b200_flac.h"
#include "ctts_b200_g711.h"

#endif /* CTTS_B200_H */
