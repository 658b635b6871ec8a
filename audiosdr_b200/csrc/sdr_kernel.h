/* sdr_kernel.h -- launcher interface between sdr_host.cpp and the kernels (sdr_kernel.cu). */
#ifndef SDR_KERNEL_H
#define SDR_KERNEL_H
#include <stdint.h>
#include "sdr_types.h"

/* state-reset bits: which reference setter side effect to replay on the device state */
enum {
  SDRK_R_IF = 1u,  /* arm_biquad_cascade_df1_init_f32 on both IF rails   (setDemodMode, C:187-222) */
  SDRK_R_IMG = 2u, /* ... on the AM image rails                           (init, C:178-179)        */
  SDRK_R_AUD = 4u, /* ... on the audio filter                             (setAudioFilter, C:298-311) */
  SDRK_R_ALS = 8u, /* taps and ring zeroed                                (enableALSfilter, C:384-391) */
  SDRK_R_NB = 16u, /* initBlanker                                         (C:676-682)              */
  /* not a setter: a channel that skipped calls of a subset (sdr_batch_process_*_subset) gets its blanker mask and ring block
   * slots turned onto the handle's block clock before its next block -- slot s moves to (s + 1) % 3 or (s + 2) % 3 (the
   * permutation of sdr_host.cpp rotate_slots).  Ignored together with SDRK_R_NB, which zeroes those slots anyway. */
  SDRK_R_TURN1 = 32u,
  SDRK_R_TURN2 = 64u
};

#ifdef __cplusplus
extern "C" {
#endif
int sdrk_setup_device(const float *hilbert64);
int sdrk_launch_pipeline(const SdrLaunch *L, void *stream);
int sdrk_launch_als_pass(const SdrLaunch *L, void *stream); /* second launch of a split ALS bucket (L->lay from lay_build_als, L->raw) */
int sdrk_occupancy(const SdrLaunch *L); /* resident CTAs per SM granted to this launch configuration (diagnostics) */
int sdrk_launch_reset(float *state, unsigned long long ch_stride, const uint32_t *chan, const uint32_t *mask, uint32_t n, void *stream);
int sdrk_launch_fill_word(float *state, unsigned long long ch_stride, uint32_t w, float v, uint32_t n_ch, void *stream);
int sdrk_launch_gather(const float *state, unsigned long long ch_stride, const uint32_t *chan, uint32_t n, const uint32_t *words,
                       uint32_t n_words, float *out, void *stream); /* words == NULL: all SDR_STATE_WORDS in order */
int sdrk_launch_scatter(float *state, unsigned long long ch_stride, const uint32_t *chan, uint32_t n, const float *in, void *stream);
#ifdef __cplusplus
}
#endif
#endif
