/*
 * ctts_b200_flac.h -- text in, one .flac file per utterance out (DESIGN.md 3.5): ctts_b200_synth_texts over a FLAC
 * session (ctts_gpu_session_begin_flac).  Exported by libctts_b200.so next to ctts_b200.h, which includes this header.
 */
#ifndef CTTS_B200_FLAC_H
#define CTTS_B200_FLAC_H

#include "ctts_front.h"
#include "ctts_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

struct ctts_b200_options;
struct ctts_b200_timing;

/* ctts_b200_synth_texts with every utterance encoded as one lossless .flac file (mono, 16 bit, at the output rate of
 * `gpu`).  out (ctts_gpu_host_alloc) holds capacity_bytes bytes; utterance u's file is out[out_offsets[u] ..
 * out_offsets[u] + out_bytes[u]) (the files are packed back to back, each starting at a multiple of 16 bytes, the
 * padding is zero) and decodes to out_counts[u] samples.  *bytes_used (may be NULL) is the space taken.  Everything
 * else as ctts_b200_synth_texts; CTTS_GPU_ERR_BOUNDS: capacity_bytes too small (ctts_b200_capacity_hint_flac). */
int ctts_b200_synth_texts_flac(ctts_front* front, ctts_gpu_ctx* gpu, const char* const* texts, const float* speeds,
                               uint32_t n, uint8_t* out, uint64_t capacity_bytes, uint64_t* out_offsets,
                               uint32_t* out_bytes, uint32_t* out_counts, uint32_t* stats, uint64_t* bytes_used,
                               const struct ctts_b200_options* opt, struct ctts_b200_timing* timing);

/* A capacity in BYTES that is enough for ctts_b200_synth_texts_flac on a context set to output rate hz: the
 * ctts_b200_capacity_hint_rate of every utterance through ctts_gpu_flac_bound, rounded up to 16.  0 for hz == 0. */
uint64_t ctts_b200_capacity_hint_flac(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n,
                                      uint32_t hz);

#ifdef __cplusplus
}
#endif

#endif /* CTTS_B200_FLAC_H */
