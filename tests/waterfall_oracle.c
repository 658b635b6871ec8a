/* tests/waterfall_oracle.c -- TEST INFRASTRUCTURE: the waterfall's definition (include/sdr_aux.h, sdr_waterfall_*) restated
 * on the host.  Each pair's power is oracle/aux_fft128.h's aux_cfft256_forward + aux_cmplx_mag_squared on the snapshot taken
 * as floats, the path of ora_grab_spectrum; the sum restarts at 0.0f, adds each pair's power in pair order with one rounding
 * per add and, after K pairs, becomes a line by one float division per bin.  The caller carries (held, acc) from one call to
 * the next, as a channel's blob does.  Compiled with the oracle's flags (-ffp-contract=off, no fast math). */
#include <stdint.h>
#include <string.h>

#include "../oracle/aux_fft128.h"

/* n_pairs snapshots [n_pairs][512] of one channel through a waterfall of K pairs per line whose state is (*held, acc[256]);
 * the completed lines go to lines[0..][256].  Returns the number of lines. */
int ora_wf_run(uint32_t K, uint32_t n_pairs, const int16_t *snaps, uint32_t *held, float *acc, float *lines) {
  int nl = 0;
  for (uint32_t j = 0; j < n_pairs; j++) {
    float buf[512], p[256];
    for (int i = 0; i < 512; i++) buf[i] = (float)snaps[(size_t)j * 512 + i];
    aux_cfft256_forward(buf);
    aux_cmplx_mag_squared(buf, p, 256);
    if (*held == 0)
      for (int b = 0; b < 256; b++) acc[b] = 0.0f;
    for (int b = 0; b < 256; b++) acc[b] = acc[b] + p[b];
    if (++*held == K) {
      for (int b = 0; b < 256; b++) lines[(size_t)nl * 256 + b] = acc[b] / (float)K;
      nl++;
      *held = 0;
    }
  }
  return nl;
}
