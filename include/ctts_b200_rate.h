/*
 * ctts_b200_rate.h -- text in, PCM out at an output rate other than 22 050 Hz (ctts_gpu_set_output_rate,
 * DESIGN.md 3.4).  Exported by libctts_b200.so next to ctts_b200.h, which includes this header.
 */
#ifndef CTTS_B200_RATE_H
#define CTTS_B200_RATE_H

#include "ctts_front.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ctts_b200_capacity_hint in samples at output rate hz: every utterance's hint converted to ceil(n * L / M)
 * samples and rounded up to 8, so it is enough for ctts_b200_synth_texts on a context set to hz.
 * ctts_b200_capacity_hint(...) == ctts_b200_capacity_hint_rate(..., 22050).  0 for hz == 0. */
uint64_t ctts_b200_capacity_hint_rate(ctts_front* front, const char* const* texts, const float* speeds, uint32_t n,
                                      uint32_t hz);

#ifdef __cplusplus
}
#endif

#endif /* CTTS_B200_RATE_H */
