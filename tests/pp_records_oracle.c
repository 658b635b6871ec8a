/* tests/pp_records_oracle.c -- TEST INFRASTRUCTURE.  The pre-processor's getters after every block, from the oracle's own
 * code: oracle/sdr_aux_oracle.c is compiled into this file unchanged, and ora_pp_run_records drives its pp_apply and
 * pp_update exactly as ora_aux_run(1, ...) does, also writing records[b][f][c] (int32 [n_blocks][6][n_channels]): the six
 * status fields (auto_detect, correction, failure_count, success_count, saved_sample, swap) of channel c right after its
 * update() for block b, before the events of block b + 1 -- what a sketch's getters return between two update() calls.
 * Built by tests/pp_records.py. */
#include "../oracle/sdr_aux_oracle.c"

int ora_pp_run_records(uint32_t n_channels, uint32_t n_blocks, const void *events, uint32_t n_events, const int16_t *in0,
                       const int16_t *in1, int16_t *out0, int16_t *out1, int32_t *records, int32_t *status) {
  const aux_event *ev = (const aux_event *)events;
  const size_t ns = (size_t)n_blocks * NB, C = n_channels;
  for (uint32_t c = 0; c < n_channels; c++) {
    pp_t p; memset(&p, 0, sizeof p);
    int16_t I[NB], Q[NB];
    for (uint32_t b = 0; b <= n_blocks; b++) {
      for (uint32_t e = 0; e < n_events; e++) /* stable order within a block; trailing events after the last block */
        if ((ev[e].channel == c || ev[e].channel == 0xFFFFFFFFu) && (b < n_blocks ? ev[e].block == b : ev[e].block >= b)) pp_apply(&p, &ev[e]);
      if (b == n_blocks) break;
      memcpy(I, in0 + c * ns + (size_t)b * NB, 2 * NB);
      memcpy(Q, in1 + c * ns + (size_t)b * NB, 2 * NB);
      pp_update(&p, I, Q);
      int32_t *r = records + (size_t)b * 6 * C + c;
      r[0] = p.autoDetectFlag; r[C] = p.I2Scorrection; r[2 * C] = p.failureCount; r[3 * C] = p.successCount;
      r[4 * C] = p.savedSample; r[5 * C] = p.IQswap;
      memcpy(out0 + c * ns + (size_t)b * NB, I, 2 * NB);
      memcpy(out1 + c * ns + (size_t)b * NB, Q, 2 * NB);
    }
    int32_t *s = status + (size_t)c * 8;
    s[0] = p.autoDetectFlag; s[1] = p.I2Scorrection; s[2] = p.failureCount; s[3] = p.successCount;
    s[4] = p.savedSample; s[5] = p.IQswap; s[6] = s[7] = 0;
  }
  return 0;
}
