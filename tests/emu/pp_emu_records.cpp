/* tests/emu/pp_emu_records.cpp -- TEST SCAFFOLDING.  The pre-processor's process call with per-block status records
 * (sdr_preproc_process_device_status) as the kernels of audiosdr_b200/csrc/sdr_aux.cu run it, on the host, from the very
 * source nvcc compiles (sdr_aux_core.cuh).  The data path is that of tests/emu/pp_emu.cpp:
 *   channels whose detector is off at the start of the call: pp_static_chunk over 8-sample chunks straight from the
 *     input planes, savedSample taken from the delayed rail afterwards (pp_static_kernel, pp_finish_kernel);
 *   the others in groups of 32 lanes (pp_detect_kernel): pp_correct_block on the staged rows, the Q15 conversion into a
 *     lane-interleaved [256][32] buffer, 7 stages of pp_fft128_stage split over PP_W warps, the power written in two
 *     phases (all reads, then all writes), pp_decide on warp 0's state, outputs with the swap.
 * and records[b][6][n_channels] = the six status fields after block b, as the records instantiations write them: for
 * channels on the feed-forward path the state at the start of the call with the saved sample moved to the delayed rail's
 * sample 128 b + 127 (pp_finish_kernel<.., true>), for the others the lane's state after pp_decide, or after
 * pp_correct_block when detection did not run in that block (pp_detect_kernel<.., true>).
 * pp_emu_run_records takes `status` as the state at the start of the call (int32 [n_channels][8]: autod, corr, fail,
 * succ, saved, swap) and writes it back at its end, so that consecutive calls continue one stream.  Events are setter calls
 * (channel, block, opcode, arg): block 0 applies before the call, as the library applies queued setters, and any later
 * block after it.
 */
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../audiosdr_b200/csrc/sdr_aux_core.cuh"
#include "../../audiosdr_b200/csrc/aux_tables.inc"

#define PP_W 8

struct Ev { uint32_t channel, block, opcode; float a0; };

static void apply_events(std::vector<PpState> &st, const Ev *ev, uint32_t n_events, bool before) {
  for (uint32_t e = 0; e < n_events; e++) {
    if ((ev[e].block == 0) != before) continue;
    for (size_t c = 0; c < st.size(); c++)
      if (ev[e].channel == c || ev[e].channel == 0xFFFFFFFFu) pp_apply(st[c], ev[e].opcode, (int32_t)ev[e].a0);
  }
}

static void record(int32_t *records, uint32_t n_channels, uint32_t b, uint32_t c, const PpState &s, int32_t saved) {
  int32_t *r = records + (size_t)b * 6 * n_channels + c;
  r[0] = s.autod; r[n_channels] = s.corr; r[2 * n_channels] = s.fail; r[3 * n_channels] = s.succ; r[4 * n_channels] = saved;
  r[5 * n_channels] = s.swap;
}

/* records: int32 [n_blocks][6][n_channels] */
extern "C" int pp_emu_run_records(uint32_t n_channels, uint32_t n_blocks, const void *events, uint32_t n_events, const int16_t *I,
                                  const int16_t *Q, int16_t *oI, int16_t *oQ, int32_t *status, int32_t *records) {
  const size_t ns = (size_t)n_blocks * 128;
  const Ev *ev = (const Ev *)events;
  std::vector<PpState> st(n_channels);
  for (uint32_t c = 0; c < n_channels; c++) {
    const int32_t *s = status + (size_t)c * 8;
    memset(&st[c], 0, sizeof(PpState));
    st[c].autod = s[0]; st[c].corr = s[1]; st[c].fail = s[2]; st[c].succ = s[3]; st[c].saved = s[4]; st[c].swap = s[5];
  }
  apply_events(st, ev, n_events, true);
  float tw[128];
  for (int k = 0; k < 128; k++) memcpy(&tw[k], &AUX_FFT_TW[k], 4);

  std::vector<uint32_t> list;
  for (uint32_t c = 0; c < n_channels; c++) {
    if (st[c].autod) { list.push_back(c); continue; }
    const PpState s = st[c]; /* pp_static_kernel: one 8-sample chunk per thread */
    const int16_t *ri = I + c * ns, *rq = Q + c * ns;
    for (uint32_t j = 0; j < n_blocks * 16; j++) {
      const size_t n = (size_t)j * 8;
      int16_t oi[8], oq[8];
      memcpy(oi, ri + n, 16); memcpy(oq, rq + n, 16);
      if (s.corr != 0) {
        int16_t pi = (int16_t)s.saved, pq = (int16_t)s.saved;
        if (j) { if (s.corr == 1) pi = ri[n - 1]; else pq = rq[n - 1]; }
        pp_static_chunk(ri + n, rq + n, pi, pq, (j & 15) == 0, s.corr, 0, oi, oq);
      }
      memcpy(oI + c * ns + n, s.swap ? oq : oi, 16);
      memcpy(oQ + c * ns + n, s.swap ? oi : oq, 16);
    }
    { /* pp_finish_kernel<.., true> */
      int32_t saved = s.saved;
      for (uint32_t b = 0; b < n_blocks; b++) {
        if (s.corr != 0) saved = (s.corr == 1 ? ri : rq)[(size_t)b * 128 + 127];
        record(records, n_channels, b, c, s, saved);
      }
    }
    if (s.corr != 0) st[c].saved = (s.corr == 1 ? ri : rq)[ns - 1]; /* pp_finish_kernel */
  }

  std::vector<float> fft(256 * 32);
  for (size_t first = 0; first < list.size(); first += 32) { /* pp_detect_kernel: one CTA = 32 listed channels */
    int16_t rowI[32][128], rowQ[32][128];
    int det[32], sw[32];
    for (uint32_t b = 0; b < n_blocks; b++) {
      for (int lane = 0; lane < 32; lane++) {
        det[lane] = 0; sw[lane] = 0;
        if (first + lane >= list.size()) continue;
        const uint32_t ch = list[first + lane];
        memcpy(rowI[lane], I + ch * ns + (size_t)b * 128, 256);
        memcpy(rowQ[lane], Q + ch * ns + (size_t)b * 128, 256);
        pp_correct_block(rowI[lane], rowQ[lane], st[ch]); /* warp 0 */
        det[lane] = st[ch].autod != 0;
        sw[lane] = st[ch].swap;
      }
      for (int w = 0; w < PP_W; w++)
        for (int lane = 0; lane < 32; lane++)
          if (det[lane])
            for (int i = w; i < 128; i += PP_W) {
              fft[(2 * i) * 32 + lane] = aux_q15_to_float(rowI[lane][i]);
              fft[(2 * i + 1) * 32 + lane] = aux_q15_to_float(rowQ[lane][i]);
            }
      for (int s = 0; s < 7; s++)
        for (int w = 0; w < PP_W; w++)
          for (int lane = 0; lane < 32; lane++)
            if (det[lane]) pp_fft128_stage(fft.data() + lane, 32, tw, s, w, PP_W);
      float pw[PP_W][32][128 / PP_W];
      for (int w = 0; w < PP_W; w++)
        for (int lane = 0; lane < 32; lane++)
          if (det[lane])
            for (int k = 0; k < 128 / PP_W; k++) pw[w][lane][k] = pp_power(fft.data() + lane, 32, w + k * PP_W);
      for (int w = 0; w < PP_W; w++)
        for (int lane = 0; lane < 32; lane++)
          if (det[lane])
            for (int k = 0; k < 128 / PP_W; k++) fft[(w + k * PP_W) * 32 + lane] = pw[w][lane][k];
      for (int lane = 0; lane < 32; lane++)
        if (det[lane]) pp_decide(fft.data() + lane, 32, st[list[first + lane]]);
      for (int lane = 0; lane < 32 && first + lane < list.size(); lane++) {
          const PpState &s = st[list[first + lane]];
          record(records, n_channels, b, list[first + lane], s, s.saved);
        }
      for (int lane = 0; lane < 32; lane++) {
        if (first + lane >= list.size()) continue;
        const uint32_t ch = list[first + lane];
        memcpy(oI + ch * ns + (size_t)b * 128, sw[lane] ? rowQ[lane] : rowI[lane], 256);
        memcpy(oQ + ch * ns + (size_t)b * 128, sw[lane] ? rowI[lane] : rowQ[lane], 256);
      }
    }
  }
  apply_events(st, ev, n_events, false);
  for (uint32_t c = 0; c < n_channels; c++) {
    int32_t *s = status + (size_t)c * 8;
    s[0] = st[c].autod; s[1] = st[c].corr; s[2] = st[c].fail; s[3] = st[c].succ; s[4] = st[c].saved; s[5] = st[c].swap;
    s[6] = s[7] = 0;
  }
  return 0;
}
