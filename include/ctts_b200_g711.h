/*
 * ctts_b200_g711.h -- text in, G.711 μ-law or A-law bytes out (DESIGN.md 3.7): ctts_b200_synth_texts over a G.711
 * session (ctts_gpu_session_begin_g711).  Exported by libctts_b200.so next to ctts_b200.h, which includes this header.
 */
#ifndef CTTS_B200_G711_H
#define CTTS_B200_G711_H

#include "ctts_front.h"
#include "ctts_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

struct ctts_b200_options;
struct ctts_b200_timing;

/* ctts_b200_synth_texts with every sample encoded as one G.711 byte of `law` (CTTS_GPU_G711_ULAW or
 * CTTS_GPU_G711_ALAW), at the output rate of `gpu` (8000 Hz for telephony: ctts_gpu_set_output_rate).  out
 * (ctts_gpu_host_alloc) holds capacity_bytes bytes; utterance u is out[out_offsets[u] .. out_offsets[u] + out_counts[u])
 * (the PCM call's packed layout with bytes in place of samples: every offset a multiple of 8, the padding holds the
 * law's code for silence).  *bytes_used (may be NULL) is the space taken.  ctts_b200_capacity_hint_rate, read as bytes,
 * is always enough; CTTS_GPU_ERR_BOUNDS: capacity_bytes too small.  Any other law is CTTS_GPU_ERR_INVALID_ARG.
 * Everything else as ctts_b200_synth_texts. */
int ctts_b200_synth_texts_g711(ctts_front* front, ctts_gpu_ctx* gpu, int law, const char* const* texts,
                               const float* speeds, uint32_t n, uint8_t* out, uint64_t capacity_bytes,
                               uint64_t* out_offsets, uint32_t* out_counts, uint32_t* stats, uint64_t* bytes_used,
                               const struct ctts_b200_options* opt, struct ctts_b200_timing* timing);

#ifdef __cplusplus
}
#endif

#endif /* CTTS_B200_G711_H */
