/* sdr_host.cpp -- host side of the C ABI (include/sdr_batch.h).
 *
 * Keeps, per channel, a shadow of the reference object's CONFIGURATION members and replays the
 * reference's setter semantics on it (which setter rebuilds which constant, which one re-initialises
 * which state: SURVEY 8a13, Q5, Q7), resolves it into the device-side SdrChanCfg with the same host
 * expressions the reference uses (so the constants are bit-equal, SURVEY N6), groups channels by
 * pipeline class into 32-lane groups, and launches the kernels.  No signal arithmetic happens here.
 *
 * C: = reference SRC/AudioSDRlib/AudioSDR.cpp, H: = .../AudioSDR.h.
 *
 * Built twice: with nvcc into the product library (CUDA backend), and with -DSDR_EMU by the test
 * suite (tests/emu) where "device" memory is host memory and the launch runs the role bodies of
 * sdr_pipeline.cuh lane by lane -- a logic check that needs no GPU, never shipped.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/sdr_batch.h"
#include "sdr_kernel.h"
#include "sdr_lay.h"
#include "sdr_tables.inc"
#include "sdr_types.h"

#ifndef SDR_EMU
#include <cuda_runtime.h>
#endif

namespace {

thread_local std::string g_err;
int fail(int code, const std::string &msg) { g_err = msg; return code; }

/* ------------------------------------------------------------------ backend */
#ifndef SDR_EMU
#define CU(call)                                                                           \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess) return fail(SDR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)
int dev_alloc(void **p, size_t n) { CU(cudaMalloc(p, n)); return 0; }
void dev_free(void *p) { if (p) cudaFree(p); }
int dev_zero(void *p, size_t n, void *s) { CU(cudaMemsetAsync(p, 0, n, (cudaStream_t)s)); return 0; }
int h2d(void *d, const void *h, size_t n, void *s) { CU(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, (cudaStream_t)s)); return 0; }
int d2h(void *h, const void *d, size_t n, void *s) { CU(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, (cudaStream_t)s)); return 0; }
int h2d_2d(void *d, size_t dp, const void *h, size_t hp, size_t w, size_t rows, void *s) {
  CU(cudaMemcpy2DAsync(d, dp, h, hp, w, rows, cudaMemcpyHostToDevice, (cudaStream_t)s)); return 0;
}
int d2h_2d(void *h, size_t hp, const void *d, size_t dp, size_t w, size_t rows, void *s) {
  CU(cudaMemcpy2DAsync(h, hp, d, dp, w, rows, cudaMemcpyDeviceToHost, (cudaStream_t)s)); return 0;
}
int dev_sync(void *s) { CU(cudaStreamSynchronize((cudaStream_t)s)); return 0; }
int dev_select(int dev) { CU(cudaSetDevice(dev)); return 0; }
int dev_stream_create(void **s) { cudaStream_t t; CU(cudaStreamCreateWithFlags(&t, cudaStreamNonBlocking)); *s = (void *)t; return 0; }
void dev_stream_destroy(void *s) { if (s) cudaStreamDestroy((cudaStream_t)s); }
int dev_event_create(void **e) { cudaEvent_t t; CU(cudaEventCreateWithFlags(&t, cudaEventDisableTiming)); *e = (void *)t; return 0; }
void dev_event_destroy(void *e) { if (e) cudaEventDestroy((cudaEvent_t)e); }
int dev_event_record(void *e, void *s) { CU(cudaEventRecord((cudaEvent_t)e, (cudaStream_t)s)); return 0; }
int dev_stream_wait(void *s, void *e) { CU(cudaStreamWaitEvent((cudaStream_t)s, (cudaEvent_t)e, 0)); return 0; }
int dev_event_sync(void *e) { CU(cudaEventSynchronize((cudaEvent_t)e)); return 0; }
#else
int dev_alloc(void **p, size_t n) { *p = calloc(1, n ? n : 1); return *p ? 0 : fail(SDR_ERR_NOMEM, "calloc"); }
void dev_free(void *p) { free(p); }
int dev_zero(void *p, size_t n, void *) { memset(p, 0, n); return 0; }
int h2d(void *d, const void *h, size_t n, void *) { memcpy(d, h, n); return 0; }
int d2h(void *h, const void *d, size_t n, void *) { memcpy(h, d, n); return 0; }
int h2d_2d(void *d, size_t dp, const void *h, size_t hp, size_t w, size_t rows, void *) {
  for (size_t r = 0; r < rows; r++) memcpy((char *)d + r * dp, (const char *)h + r * hp, w); return 0;
}
int d2h_2d(void *h, size_t hp, const void *d, size_t dp, size_t w, size_t rows, void *) {
  for (size_t r = 0; r < rows; r++) memcpy((char *)h + r * hp, (const char *)d + r * dp, w); return 0;
}
int dev_sync(void *) { return 0; }
int dev_select(int) { return 0; }
int dev_stream_create(void **s) { *s = nullptr; return 0; }
void dev_stream_destroy(void *) {}
int dev_event_create(void **e) { *e = nullptr; return 0; }
void dev_event_destroy(void *) {}
int dev_event_record(void *, void *) { return 0; }
int dev_stream_wait(void *, void *) { return 0; }
int dev_event_sync(void *) { return 0; }
#endif

inline float tabf(const uint32_t *t, int i) { float f; memcpy(&f, &t[i], 4); return f; }

const float FS = SDR_SAMPLE_RATE;
const double PI_D = 3.1415926535897932384626433832795; /* Arduino PI */
const float IF_CENTER = 6890.0f, BW_SSB = 3000.0f, BW_CW = 1000.0f, BW_WSPR = 1000.0f, BW_AM = 8500.0f; /* H:164-168 */

/* ------------------------------------------------------------------ per-channel shadow of the reference's configuration */
struct Shadow {
  int mode; float freq_shift; bool muted;
  float in_gain, in_gain_i, in_gain_q, gain_balance, out_gain;
  bool aud_on; int aud_id; int aud_set; int if_set;
  int als_m, als_delay; float als_lambda; bool als_on, als_notch, als_adapt;
  float thr, slope, knee, t_att, t_rel, t_hang, a_att, b_att, a_rel, b_rel, static_gain; uint32_t hang_count; bool agc_on;
  int lut_id;
  float nb_thr; bool nb_on;
};

struct AgcKey {
  uint32_t a, b, c;
  bool operator<(const AgcKey &o) const { return a != o.a ? a < o.a : (b != o.b ? b < o.b : c < o.c); }
};
inline uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

/* H:483-491 */
float log2_approx(float v) {
  int e; float m = frexpf(fabsf(v), &e);
  return (((1.23149591368684f * m - 4.11852516267426f) * m + 6.02197014179219f) * m - 3.13396450166353f) + e;
}
/* agc_createLookupTable, C:459-480.  130 entries are computed (the reference writes one past its
 * 129-float array, SURVEY Q8); the hot path reads entries 0..128 only. */
void build_agc_lut(float thr, float slope, float knee, float *lut) {
  float lo = expf(2.3025 * (thr - knee / 2.0) / 20.0);
  float hi = expf(2.3025 * (thr + knee / 2.0) / 20.0);
  for (int i = 0; i < 130; i++) {
    float in = (float)i / 128.0;
    float in_db = 6.026 * log2_approx(in);
    if (in < lo) lut[i] = 1.0;
    else if (in > hi) { float out_db = (thr + (in_db - thr) * slope); lut[i] = expf(2.3025 * (out_db - in_db) / 20.0); }
    else {
      float out_db = in_db + ((slope - 1.0) * (in_db - thr + knee / 2.0) * (in_db - thr + knee / 2.0)) / (2.0 * knee);
      lut[i] = expf(2.3025 * (out_db - in_db) / 20.0);
    }
  }
  lut[130] = lut[131] = 0.0f;
}

/* the blanker's mask words and ring planes are indexed by (absolute block index % 3): moving a channel between handles
 * that have processed different numbers of blocks turns the slots by the difference */
void rotate_slots(float *w, uint32_t delta) {
  if (delta % 3 == 0) return;
  std::vector<float> t(w, w + SDR_STATE_WORDS);
  for (uint32_t s = 0; s < 3; s++) {
    const uint32_t d = (s + delta) % 3;
    memcpy(w + W_NB_MASK + d * 32, &t[W_NB_MASK + s * 32], 32 * sizeof(float));
    for (uint32_t pl = 0; pl < 3; pl++) memcpy(w + W_NB_RING + pl * 384 + d * 128, &t[W_NB_RING + pl * 384 + s * 128], 128 * sizeof(float));
  }
}
}  // namespace

/* the groups of one pipeline class with one set of optional stages: one kernel launch with its own shared-memory plan */
struct Bucket {
  SdrLay lay; uint32_t first, count;
  /* a bucket with the ALS filter and more groups than SMs runs as two launches (sdr_lay.h, lay_build_als): the chain up to
   * the AGC on the plan the bucket would have without ALS, then the ALS + output post-pass, four groups to an SM */
  bool split; SdrLay lay_main, lay_als;
};

/* the groups and buckets of one set of channels: every channel of the handle, or the channels of a subset call */
struct Grouping {
  std::vector<SdrGroup> groups; std::vector<Bucket> buckets;
  SdrGroup *d_groups; size_t cap;
};

enum { SDR_HOST_TICKETS = 8 }; /* host calls whose completion can be waited for one by one (sdr_batch_wait_host_ticket) */
enum { SDR_MAX_BUCKETS = 12 }; /* SSB class: blanker x ALS = 4; ENV class: blanker x ALS x SAM-only = 8 */

struct sdr_batch {
  sdr_batch_desc desc;
  std::vector<Bucket> buckets;
  void *s_aux[SDR_MAX_BUCKETS]; void *ev_fork, *ev_join[SDR_MAX_BUCKETS]; /* buckets beyond the first run on their own streams, forked from / joined to the caller's */
  uint32_t n_ch; size_t ch_stride;
  std::vector<Shadow> sh;
  std::vector<uint32_t> pend_reset; /* per channel SDRK_R_* bits to replay before the next block */
  std::vector<uint32_t> dirty_list;
  std::vector<uint32_t> cfg_list; std::vector<uint8_t> cfg_mark; bool cfg_all; /* channels whose setters ran since the last sync (cfg_all: every one) */
  bool cfg_dirty, groups_dirty, luts_dirty;
  std::map<AgcKey, int> lut_index;
  std::vector<float> luts; /* [n][SDR_AGC_LUT_STRIDE] */
  size_t lut_gc_at; /* registry size at which unused tables are looked for next (collect_luts) */
  /* device */
  float *d_state; SdrChanCfg *d_cfg; float *d_luts; SdrTables *d_tabs;
  uint32_t *d_reset_ch, *d_reset_mask; size_t reset_cap; size_t luts_cap;
  float *d_gather; uint32_t *d_gather_ids; uint32_t *d_gather_words; size_t gather_cap;
  /* host-buffer path: two staging sets and three streams so that the H2D copy of chunk k+1, the kernel of chunk k and
   * the D2H copy of chunk k-1 overlap */
  void *d_in_i[2], *d_in_q[2], *d_out[2]; size_t stage_in_bytes, stage_out_bytes;
  void *d_bs[2]; size_t stage_bs_bytes; /* per-block status records of a chunk, beside d_out (allocated by the first call that asks for records) */
  void *s_h2d, *s_comp, *s_d2h; void *ev_h2d[2], *ev_comp[2], *ev_d2h[2];
  uint64_t host_seq; /* chunks queued by submit_host since create: chunk n uses staging set n & 1 */
  uint64_t host_calls; void *ev_call[SDR_HOST_TICKETS]; /* host calls queued since create (= the ticket of the latest); call t's last copy-out records ev_call[t % SDR_HOST_TICKETS] */
  float *d_raw[SDR_MAX_BUCKETS]; size_t raw_cap[SDR_MAX_BUCKETS]; /* scratch planes of split ALS buckets (by bucket index), grown on demand */
  unsigned long long *d_prof; size_t prof_cap; bool prof_on; uint64_t prof_launches;
  std::vector<uint64_t> prof_busy, prof_total, prof_groups, prof_extra, prof_load, prof_crit, prof_bar; /* folded per class */
  uint64_t blocks_done, launches;
  void *last_stream;
  std::vector<SdrChanCfg> h_cfg;
  /* every channel (the plain calls), and the last subset call's channels: kept apart, so that alternating the two forms
   * re-plans neither; the subset grouping is reused while its id list and the configuration stay the same */
  Grouping all, sub;
  std::vector<uint32_t> sub_ids; bool sub_valid;
  int prof_of; /* the grouping the profile rows belong to: 0 all, 1 sub */
  /* Block clocks.  The blanker slots of a channel are laid out for the handle's block clock after the last call that ran
   * it (or the import that installed it): max(plain_at, at[c]).  A channel whose layout is behind the clock when a call
   * lists it again is turned first (SDRK_R_TURN*).  own[c]: the channel's blocks in subset calls (it has also run every
   * block of the plain calls), the order of a subset's channels inside a bucket. */
  uint64_t plain_at; bool sub_since_plain;
  std::vector<uint64_t> at, own;
  std::vector<uint8_t> id_mark;
};

namespace {

int lut_for(sdr_batch *h, float thr, float slope, float knee) {
  AgcKey k{fbits(thr), fbits(slope), fbits(knee)};
  auto it = h->lut_index.find(k);
  if (it != h->lut_index.end()) return it->second;
  int id = (int)(h->luts.size() / SDR_AGC_LUT_STRIDE);
  h->luts.resize(h->luts.size() + SDR_AGC_LUT_STRIDE);
  build_agc_lut(thr, slope, knee, &h->luts[(size_t)id * SDR_AGC_LUT_STRIDE]);
  h->lut_index[k] = id;
  h->luts_dirty = true;
  return id;
}

/* setDemodMode, C:187-222: sets _freq_shift and re-initialises BOTH IF cascades (state zeroed); nothing else */
int set_mode(sdr_batch *h, uint32_t c, int m) {
  Shadow &s = h->sh[c];
  if (m < 0 || m > 6) return fail(SDR_ERR_MODE, "setDemodMode: mode outside 0..6");
  int old_cls = (s.mode == SDR_AM || s.mode == SDR_SAM) ? CLS_ENV : CLS_SSB;
  s.mode = m;
  if (m == SDR_USB) { s.freq_shift = IF_CENTER - BW_SSB / 2.0; s.if_set = 0; }
  else if (m == SDR_LSB) { s.freq_shift = IF_CENTER + BW_SSB / 2.0; s.if_set = 0; }
  else if (m == SDR_WSPR) { s.freq_shift = IF_CENTER - BW_SSB / 2.0; s.if_set = 2; }
  else if (m == SDR_CW_USB) { s.freq_shift = IF_CENTER - BW_CW / 2.0; s.if_set = 1; }
  else if (m == SDR_CW_LSB) { s.freq_shift = IF_CENTER + BW_CW / 2.0; s.if_set = 1; }
  else { s.freq_shift = IF_CENTER; s.if_set = 3; }
  h->pend_reset[c] |= SDRK_R_IF;
  int cls = (m == SDR_AM || m == SDR_SAM) ? CLS_ENV : CLS_SSB;
  if (cls != old_cls) h->groups_dirty = true;
  return 0;
}

void agc_attack(Shadow &s, float ms) { s.t_att = ms; s.a_att = exp(log(0.1) / (FS * s.t_att / 1000.0)); s.b_att = 1.0 - s.a_att; }   /* C:551-555 */
void agc_release(Shadow &s, float ms) { s.t_rel = ms; s.a_rel = exp(log(0.1) / (FS * s.t_rel / 1000.0)); s.b_rel = 1.0 - s.a_rel; } /* C:557-561 */
void agc_hang(Shadow &s, float ms) { s.t_hang = ms; s.hang_count = s.t_hang * FS / 1000.0; }                                         /* C:563-566 */

/* init(), C:174-185 */
void do_init(sdr_batch *h, uint32_t c) {
  Shadow &s = h->sh[c];
  s.aud_set = SDR_AUDIO_2700;
  /* agc_init, C:439-457 */
  s.thr = -60.0; s.slope = 0.1; s.knee = 2.0; s.t_att = 5.0; s.t_rel = 500.0; s.t_hang = 100.0;
  s.hang_count = FS * (s.t_hang / 1000.0);
  s.a_att = exp(log(0.1) / (FS * s.t_att / 1000.0)); s.b_att = 1.0 - s.a_att;
  s.a_rel = exp(log(0.1) / (FS * s.t_rel / 1000.0)); s.b_rel = 1.0 - s.a_rel;
  s.agc_on = true;
  s.lut_id = lut_for(h, s.thr, s.slope, s.knee);
  h->pend_reset[c] |= SDRK_R_AUD | SDRK_R_IF | SDRK_R_IMG | SDRK_R_NB;
  set_mode(h, c, SDR_LSB);
  s.muted = false;
}

/* constructor defaults, H:164-284 (members never initialised there read as zero, SURVEY Q4) */
void construct(sdr_batch *h, uint32_t c) {
  Shadow &s = h->sh[c];
  memset(&s, 0, sizeof s);
  s.in_gain = s.in_gain_i = s.in_gain_q = s.gain_balance = 1.0f; s.out_gain = 0.5; s.muted = true;
  s.als_m = 55; s.als_delay = 3; s.als_lambda = 0.5; s.als_on = false; s.als_notch = true; s.als_adapt = true;
  s.static_gain = 10.0; s.agc_on = true;
  s.nb_thr = 1.2; s.nb_on = true;
  s.aud_on = false; s.aud_id = 0;
  do_init(h, c);
}

int apply_one(sdr_batch *h, uint32_t c, uint32_t op, float a0, float a1, float a2) {
  Shadow &s = h->sh[c];
  switch (op) {
    case SDR_SET_setMute: s.muted = (a0 != 0.0f); break;
    case SDR_SET_setInputGain: { float g = a0; if (g > 10.0) g = 10.0; if (g < 0.0) g = 0.0;
      s.in_gain = g; s.in_gain_i = s.in_gain * s.gain_balance; s.in_gain_q = s.in_gain; } break;
    case SDR_SET_setIQgainBalance: { float bal = sqrtf(a0); /* a LOCAL in the reference: the member stays 1 (Q7) */
      s.in_gain_i = s.in_gain * bal; s.in_gain_q = s.in_gain / bal; } break;
    case SDR_SET_setDemodMode: { int rc = set_mode(h, c, (int)a0); if (rc) return rc; } break; /* falls through to cfg_dirty: mode, phase increment and IF set are device configuration */
    case SDR_SET_enableAudioFilter: s.aud_on = true; break;
    case SDR_SET_disableAudioFilter: s.aud_on = false; break;
    case SDR_SET_setOutputGain: s.out_gain = a0; break;
    case SDR_SET_setAudioFilter: { int id = (int)a0;
      if (id < 0 || id > SDR_AUDIO_BYPASS) return fail(SDR_ERR_MODE, "setAudioFilter: id outside 0..10");
      if (id == SDR_AUDIO_BYPASS) s.aud_on = false;
      else { s.aud_set = id; h->pend_reset[c] |= SDRK_R_AUD; }
      s.aud_id = id; } break;
    case SDR_SET_enableALSfilter: s.als_on = true; h->pend_reset[c] |= SDRK_R_ALS; break;
    case SDR_SET_disableALSfilter: s.als_on = false; break;
    case SDR_SET_setALSfilterNotch: s.als_notch = true; break;
    case SDR_SET_setALSfilterPeak: s.als_notch = false; break;
    case SDR_SET_setALSfilterAdaptive: s.als_adapt = true; break;
    case SDR_SET_setALSfilterStatic: s.als_adapt = false; break;
    case SDR_SET_setALSfilterParams: {
      int m = (int16_t)(unsigned)a0; if (m >= SDR_BLOCK_SAMPLES) m = SDR_BLOCK_SAMPLES;
      int d = (int16_t)a2;
      /* the reference indexes _als_in[(i - delay) - j] with i >= 128: anything reaching below 0 is out of bounds there */
      if (m < 0 || d < 0 || m + d > 129) return fail(SDR_ERR_UNSUPPORTED, "setALSfilterParams: M + delay > 129 or negative");
      s.als_m = m; s.als_lambda = a1; s.als_delay = d; } break;
    case SDR_SET_enableAGC: s.agc_on = true; break;
    case SDR_SET_disableAGC: s.agc_on = false; break;
    case SDR_SET_setAGCthreshold: s.thr = a0; s.lut_id = lut_for(h, s.thr, s.slope, s.knee); break;
    case SDR_SET_setAGCslope: s.slope = a0; s.lut_id = lut_for(h, s.thr, s.slope, s.knee); break;
    case SDR_SET_setAGCmode: { int m = (int16_t)a0;
      if (m < 0 || m > 3) return fail(SDR_ERR_MODE, "setAGCmode: mode outside 0..3");
      if (m == SDR_AGC_OFF) s.agc_on = false;
      else if (m == SDR_AGC_FAST) { agc_attack(s, 2.0); agc_release(s, 100.0); agc_hang(s, 100.0); s.agc_on = true; }
      else if (m == SDR_AGC_MEDIUM) { agc_attack(s, 5.0); agc_release(s, 250.0); agc_hang(s, 500.0); s.agc_on = true; }
      else { agc_attack(s, 10.0); agc_release(s, 500.0); agc_hang(s, 2000.0); s.agc_on = true; } } break;
    case SDR_SET_setAGCkneeWidth: s.knee = a0; s.lut_id = lut_for(h, s.thr, s.slope, s.knee); break;
    case SDR_SET_setAGCattackTime: agc_attack(s, a0); break;
    case SDR_SET_setAGCreleaseTime: agc_release(s, a0); break;
    case SDR_SET_setAGChangTime: agc_hang(s, a0); break;
    case SDR_SET_setAGCstaticGain: s.static_gain = a0; break;
    case SDR_SET_enableNoiseBlanker: s.nb_on = true; h->pend_reset[c] |= SDRK_R_NB; break;
    case SDR_SET_disableNoiseBlanker: s.nb_on = false; break;
    case SDR_SET_setNoiseBlankerThreshold: s.nb_thr = a0; h->pend_reset[c] |= SDRK_R_NB; break;
    case SDR_SET_setNoiseBlankerThresholdDb: s.nb_thr = powf(10.0, (a0 / 20.0)); h->pend_reset[c] |= SDRK_R_NB; break;
    case SDR_SET_init: do_init(h, c); break;
    default: return fail(SDR_ERR_ARG, "unknown setter id");
  }
  h->cfg_dirty = true;
  if (!h->cfg_all && !h->cfg_mark[c]) {
    h->cfg_mark[c] = 1; h->cfg_list.push_back(c);
    if (h->cfg_list.size() > h->n_ch / 4 + 64) { h->cfg_all = true; for (uint32_t k : h->cfg_list) h->cfg_mark[k] = 0; h->cfg_list.clear(); }
  }
  return 0;
}

void resolve(const Shadow &s, SdrChanCfg &c) {
  memset(&c, 0, sizeof c);
  c.mode = s.mode;
  c.flags = (s.nb_on ? CF_NB : 0) | (s.aud_on ? CF_AUD : 0) | (s.agc_on ? CF_AGC : 0) | (s.als_on ? CF_ALS : 0) |
            (s.als_notch ? CF_ALS_NOTCH : 0) | (s.als_adapt ? CF_ALS_ADAPT : 0) | (s.muted ? CF_MUTED : 0);
  c.in_gain_i = s.in_gain_i; c.in_gain_q = s.in_gain_q; c.out_gain = s.out_gain;
  const float two_pi = (float)(2.0 * PI_D);
  c.ssb_phase_inc = (-s.freq_shift) * (two_pi / FS); /* freq_shifter's phase_inc, H:510, with freq_shift = -_freq_shift (C:86) */
  c.if_set = s.if_set; c.aud_set = s.aud_set;
  c.agc_a_att = s.a_att; c.agc_b_att = s.b_att; c.agc_a_rel = s.a_rel; c.agc_b_rel = s.b_rel; c.agc_static_gain = s.static_gain;
  c.agc_hang_count = s.hang_count; c.agc_lut = s.lut_id;
  c.nb_thr = s.nb_thr; c.als_m = s.als_m; c.als_delay = s.als_delay; c.als_lambda = s.als_lambda;
}

uint32_t lay_feat_of(uint32_t flags) { return ((flags & CF_NB) ? LF_NB : 0u) | ((flags & CF_ALS) ? LF_ALS : 0u); }

int env_int(const char *name, int dflt) { const char *e = getenv(name); return e && *e ? atoi(e) : dflt; }

/* Tile length and shared-memory budget of a bucket.  A group's time does not depend on how many other groups run, so
 * when a launch has more groups than SMs the plan trades ring slack for co-residency: shorter tiles shrink every ring
 * that is sized in tiles.  (SDR_TILE_SSB / SDR_TILE_ENV / SDR_CTAS_PER_SM / SDR_SLACK override the choice for experiments.) */
int plan_bucket(Bucket &b, int cls, uint32_t feat, int n_sm, uint32_t handle_groups) {
  /* Measured (DESIGN.md section 7): the SSB class is bound by its four Hilbert warps per SM whatever the tile length, so it
   * stays on the 32-sample plan; an ENV group is bound by the latency of its one PLL warp, so ENV buckets without blanker
   * and ALS run 16-sample tiles in a fraction of the shared memory -- two groups per SM; SAM-only buckets with the light
   * stages merged (7 warps) three groups per SM -- when there are enough groups to share. */
  int T = 32, ctas = 1, in_depth = 0;
  const bool lean = !(feat & (LF_NB | LF_ALS));
  if (cls == CLS_ENV && lean && b.count > (uint32_t)n_sm) {
    if ((feat & LF_SAM) && b.count > 2u * (uint32_t)n_sm) { T = 16; ctas = 3; in_depth = 1; } /* 76.7 KB: three fit an SM exactly */
    else {
      /* at most two groups per SM: the 11-warp plan spreads a group over more warps than the merged one and is the faster of
       * the two while the SM is not crowded (8 192 SAM channels = the shard of one of eight GPUs: 40.6 against 37.3 G, run r02z) */
      T = 16; ctas = 2; feat &= ~(uint32_t)LF_SAM;
    }
  }
  const int t_env = env_int(cls == CLS_SSB ? "SDR_TILE_SSB" : "SDR_TILE_ENV", 0);
  if (t_env && lean) { T = t_env; ctas = T == 32 ? 1 : 2; in_depth = 0; }
  const int c_env = env_int("SDR_CTAS_PER_SM", 0);
  if (c_env > 0) ctas = c_env;
  if (env_int("SDR_NO_MERGE", 0)) feat &= ~(uint32_t)LF_SAM;
  const int slack = env_int("SDR_SLACK", 0); /* extra ring slots only matter to the hand-over build (-DSDR_HANDOVER) */
  const int budget = (233472 - 1024 * ctas) / ctas; /* an SM has 228 KB, each resident CTA costs 1 KB of it */
  /* experiments: input requests ahead (SDR_IN_DEPTH), order of the merged plan's seven warp programs (SDR_MAP_ENV_MERGED: a
   * permutation of 0..6 as hex digits, warp 0 first; programs: 0 in+out, 1 IF-I, 2 IF-Q, 3 PLL, 4 envelope path, 5 audio, 6 AGC) */
  uint8_t mo[7]; const uint8_t *merged_order = nullptr;
  if (const char *e = getenv("SDR_MAP_ENV_MERGED")) {
    unsigned seen = 0;
    if (strlen(e) == 7) for (int w = 0; w < 7; w++) { mo[w] = (uint8_t)(e[w] - '0'); if (mo[w] < 7) seen |= 1u << mo[w]; }
    if (seen == 0x7Fu) merged_order = mo;
  }
  int rc = lay_build_ex(&b.lay, cls, feat, T, budget > 232448 ? 232448 : budget, slack, env_int("SDR_IN_DEPTH", in_depth), merged_order);
  if (rc) rc = lay_build(&b.lay, cls, feat, 32, 232448, 0);
  if (rc) return rc;
  /* measured placements */
  if (b.lay.n_warps == SDR_STAGES) {
    unsigned long long m = cls == CLS_SSB ? ((feat & LF_ALS) ? SDR_MAP_SSB_ALS_DEFAULT : (feat & LF_NB) ? SDR_MAP_SSB_DEFAULT : SDR_MAP_SSB_NONB_DEFAULT)
                                          : ((feat & LF_NB) && !(feat & LF_ALS) ? SDR_MAP_ENV_NB_DEFAULT : SDR_MAP_ENV_DEFAULT);
    if (const char *e = getenv(cls == CLS_SSB ? "SDR_MAP_SSB" : "SDR_MAP_ENV")) m = strtoull(e, nullptr, 16);
    lay_place(&b.lay, m);
  } else if (cls == CLS_ENV && b.lay.n_warps == 11) {
    unsigned long long m = SDR_MAP_ENV_LEAN_DEFAULT;
    if (const char *e = getenv("SDR_MAP_ENV_LEAN")) m = strtoull(e, nullptr, 16);
    lay_place(&b.lay, m);
  } else if (const char *e = getenv("SDR_MAP_SSB_LEAN")) lay_place(&b.lay, strtoull(e, nullptr, 16));
  /* ALS buckets: one launch while every group of the handle has an SM to itself (the ALS warp then runs beside the chain at
   * no cost in waves); two launches beyond that (the buckets of a handle run side by side and share the SMs, so the handle's
   * group count decides).  SDR_ALS_SPLIT=0 / 1 forces one form (tests, A/B runs). */
  b.split = false;
  const int sp = env_int("SDR_ALS_SPLIT", -1);
  if ((feat & LF_ALS) && sp != 0 && (handle_groups > (uint32_t)n_sm || sp == 1)) {
    Bucket m; m.first = b.first; m.count = b.count;
    if (plan_bucket(m, cls, feat & ~(uint32_t)LF_ALS, n_sm, handle_groups) == 0) { b.lay_main = m.lay; b.split = true; } /* (lay_als: build_groups) */
  }
  return 0;
}

/* Groups and buckets of the channels ids[0..n) (ids == nullptr: every channel), lane rows = the channels' positions in the
 * list (their ids for every channel), with each group's feature summary and staged AGC tables. */
int build_groups(sdr_batch *h, Grouping &G, const uint32_t *ids, uint32_t n) {
  G.groups.clear(); G.buckets.clear();
  /* Channels of one class with the same optional stages share groups (= one bucket, one launch); inside a bucket they are
   * ordered by mode so that the lanes of a warp run the same oscillator frequency and coefficient set (channel results
   * never depend on the grouping).  A subset's channels are also ordered by blocks processed: lanes with the same history
   * keep one oscillator phase, so RoleNco stays on its one-oscillator table path. */
  static const int order[2][5] = {{SDR_LSB, SDR_USB, SDR_CW_LSB, SDR_CW_USB, SDR_WSPR}, {SDR_AM, SDR_SAM, -1, -1, -1}};
  std::vector<uint32_t> by_key[2][8][5]; /* positions in the list */
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = ids ? ids[i] : i;
    const int m = h->sh[c].mode, cls = (m == SDR_AM || m == SDR_SAM) ? CLS_ENV : CLS_SSB;
    int mi = 0;
    for (int k = 0; k < 5; k++) if (order[cls][k] == m) mi = k;
    uint32_t f = lay_feat_of(h->h_cfg[c].flags);
#ifndef SDR_HANDOVER
    if (m == SDR_SAM) f |= LF_SAM; /* SAM channels get groups (and a bucket) of their own: no AM lane among them */
#endif
    by_key[cls][f][mi].push_back(i);
  }
  if (ids)
    for (auto &a : by_key) for (auto &b : a) for (auto &v : b)
      std::stable_sort(v.begin(), v.end(), [&](uint32_t x, uint32_t y) { return h->own[ids[x]] < h->own[ids[y]]; });
  for (int cls = 0; cls < 2; cls++) {
    for (uint32_t feat = 0; feat < 8; feat++) {
      Bucket b; b.first = (uint32_t)G.groups.size();
      SdrGroup g; int fill = 0;
      auto flush = [&]() {
        if (!fill) return;
        for (int l = fill; l < SDR_LANES; l++) g.cid[l] = g.row[l] = -1;
        G.groups.push_back(g); fill = 0;
      };
      for (int mi = 0; mi < 5; mi++) {
        for (uint32_t i : by_key[cls][feat][mi]) {
          if (!fill) { memset(&g, 0, sizeof g); g.cls = cls; }
          g.cid[fill] = (int32_t)(ids ? ids[i] : i); g.row[fill] = (int32_t)i; fill++;
          if (fill == SDR_LANES) flush();
        }
        /* SSB class: a group never mixes modes, so that all its lanes share one oscillator (RoleNco's table path) */
        if (cls == CLS_SSB) flush();
      }
      flush();
      b.count = (uint32_t)G.groups.size() - b.first;
      if (!b.count) continue;
      b.lay.cls = cls; b.lay.feat = feat; /* planned below, when the grouping's group count is known */
      G.buckets.push_back(b);
    }
  }
  const uint32_t n_groups = (uint32_t)G.groups.size();
  if (G.buckets.size() > (size_t)SDR_MAX_BUCKETS) return fail(SDR_ERR_UNSUPPORTED, "more buckets than SDR_MAX_BUCKETS (internal)");
  for (Bucket &b : G.buckets) {
    if (plan_bucket(b, b.lay.cls, b.lay.feat, 148, n_groups)) return fail(SDR_ERR_UNSUPPORTED, "no shared-memory plan for a bucket (internal)");
    if (b.split) { /* the post-pass keeps as many taps and as much input history as the bucket's channels ask for (C:393-398) */
      int m_max = 0, reach_max = 0;
      for (uint32_t g = b.first; g < b.first + b.count; g++)
        for (int l = 0; l < SDR_LANES; l++) {
          const int c = G.groups[g].cid[l];
          if (c < 0 || !(h->h_cfg[c].flags & CF_ALS)) continue;
          const SdrChanCfg &k = h->h_cfg[c];
          m_max = std::max(m_max, (int)k.als_m); reach_max = std::max(reach_max, (int)k.als_m + (int)k.als_delay);
        }
      if (env_int("SDR_ALS_FULL_ROWS", 0)) { m_max = 128; reach_max = 129; } /* experiment / tests: the largest plan whatever the parameters */
      if (lay_build_als(&b.lay_als, m_max, reach_max)) return fail(SDR_ERR_UNSUPPORTED, "no plan for the ALS post-pass (internal)");
      if (env_int("SDR_ALS_NO_MIRROR", 0) && b.lay_als.als_mirror) { b.lay_als.als_mirror = 0; b.lay_als.smem_bytes -= b.lay_als.nc * b.lay_als.tile_f * 4; }
    }
  }
  for (SdrGroup &g : G.groups) {
    g.feat = 0;
    for (int k = 0; k < SDR_LUT_SLOTS; k++) g.lut_ids[k] = -1;
    for (int l = 0; l < SDR_LANES; l++) {
      g.lut_slot[l] = 255;
      if (g.cid[l] < 0) continue;
      g.feat |= h->h_cfg[g.cid[l]].flags;
      int id = h->h_cfg[g.cid[l]].agc_lut;
      for (int k = 0; k < SDR_LUT_SLOTS; k++) {
        if (g.lut_ids[k] == id) { g.lut_slot[l] = (uint8_t)k; break; }
        if (g.lut_ids[k] < 0) { g.lut_ids[k] = id; g.lut_slot[l] = (uint8_t)k; break; }
      }
      if (g.lut_slot[l] == 255) g.feat |= GF_LUT_GLOBAL;
    }
  }
  return 0;
}

/* The grouping's groups to the device, in stream order: a launch of an earlier call that reads the buffer was queued on
 * `stream` or joined into it (a buffer that must grow waits for the handle's last stream before it is freed). */
int upload_groups(sdr_batch *h, Grouping &G, void *stream) {
  size_t need = sizeof(SdrGroup) * std::max<size_t>(G.groups.size(), 1);
  if (need > G.cap) {
    if (G.d_groups) { if (dev_sync(h->last_stream)) return SDR_ERR_CUDA; dev_free(G.d_groups); G.d_groups = nullptr; G.cap = 0; }
    if (dev_alloc((void **)&G.d_groups, need)) return SDR_ERR_NOMEM;
    G.cap = need;
  }
  if (!G.groups.empty() && h2d(G.d_groups, G.groups.data(), sizeof(SdrGroup) * G.groups.size(), stream)) return SDR_ERR_CUDA;
  return 0;
}

int fold_profile(sdr_batch *h);

/* AGC tables nobody uses any more (a sweep of setAGCthreshold / slope / kneeWidth leaves one behind per step): when the
 * registry has doubled since the last look, keep the tables some channel still points to and renumber them */
void collect_luts(sdr_batch *h) {
  const size_t n = h->luts.size() / SDR_AGC_LUT_STRIDE;
  if (n <= h->lut_gc_at) return;
  std::vector<int> remap(n, -1);
  size_t used = 0;
  for (const Shadow &s : h->sh) if (remap[s.lut_id] < 0) remap[s.lut_id] = (int)used++;
  if (used < n) {
    std::vector<float> kept(used * SDR_AGC_LUT_STRIDE);
    for (size_t i = 0; i < n; i++) if (remap[i] >= 0) memcpy(&kept[(size_t)remap[i] * SDR_AGC_LUT_STRIDE], &h->luts[i * SDR_AGC_LUT_STRIDE], sizeof(float) * SDR_AGC_LUT_STRIDE);
    h->luts.swap(kept);
    for (auto it = h->lut_index.begin(); it != h->lut_index.end();) { if (remap[it->second] < 0) it = h->lut_index.erase(it); else { it->second = remap[it->second]; ++it; } }
    for (Shadow &s : h->sh) s.lut_id = remap[s.lut_id];
    h->luts_dirty = h->cfg_dirty = h->cfg_all = true;
  }
  h->lut_gc_at = std::max<size_t>(64, 2 * used);
}

int sync_config(sdr_batch *h, void *stream) {
  collect_luts(h);
  if (h->luts_dirty) {
    size_t need = h->luts.size() * sizeof(float);
    if (need > h->luts_cap) {
      if (h->d_luts) { if (dev_sync(h->last_stream)) return SDR_ERR_CUDA; dev_free(h->d_luts); }
      size_t cap = std::max(need * 2, (size_t)SDR_AGC_LUT_STRIDE * 4 * 16);
      if (dev_alloc((void **)&h->d_luts, cap)) return SDR_ERR_NOMEM;
      h->luts_cap = cap;
    }
    if (h2d(h->d_luts, h->luts.data(), need, stream)) return SDR_ERR_CUDA;
    h->luts_dirty = false;
  }
  if (h->cfg_dirty) {
    if (h->cfg_all) {
      for (uint32_t c = 0; c < h->n_ch; c++) resolve(h->sh[c], h->h_cfg[c]);
      if (h2d(h->d_cfg, h->h_cfg.data(), sizeof(SdrChanCfg) * h->n_ch, stream)) return SDR_ERR_CUDA;
      h->groups_dirty = true; /* group feature summaries depend on the flags */
    } else {
      /* only the channels whose setters ran: re-resolve them, upload the span they cover (or each one, when they are few
       * and far apart), and plan the groups again only if something the grouping depends on has changed */
      uint32_t lo = h->n_ch, hi = 0;
      for (uint32_t c : h->cfg_list) {
        const SdrChanCfg old = h->h_cfg[c];
        resolve(h->sh[c], h->h_cfg[c]);
        const SdrChanCfg &now = h->h_cfg[c];
        if (old.mode != now.mode || old.flags != now.flags || old.agc_lut != now.agc_lut || old.als_m != now.als_m || old.als_delay != now.als_delay)
          h->groups_dirty = true;
        lo = std::min(lo, c); hi = std::max(hi, c);
        h->cfg_mark[c] = 0;
      }
      if (!h->cfg_list.empty()) {
        if (h->cfg_list.size() <= 16 && (size_t)(hi - lo + 1) > 64 * h->cfg_list.size()) {
          for (uint32_t c : h->cfg_list) if (h2d(h->d_cfg + c, &h->h_cfg[c], sizeof(SdrChanCfg), stream)) return SDR_ERR_CUDA;
        } else if (h2d(h->d_cfg + lo, &h->h_cfg[lo], sizeof(SdrChanCfg) * (hi - lo + 1), stream)) return SDR_ERR_CUDA;
      }
    }
    for (uint32_t c : h->cfg_list) h->cfg_mark[c] = 0; /* (also when cfg_all was raised with channels already listed) */
    h->cfg_list.clear(); h->cfg_all = false;
    h->cfg_dirty = false;
  }
  if (h->groups_dirty) {
    if (h->prof_on && fold_profile(h)) return SDR_ERR_CUDA; /* rows are per group: fold before the grouping changes */
    { int rc = build_groups(h, h->all, nullptr, h->n_ch); if (rc) return rc; }
    { int rc = upload_groups(h, h->all, stream); if (rc) return rc; }
    h->sub_valid = false; /* (built from the same configuration) */
    h->groups_dirty = false;
  }
  /* replay pending state re-initialisations */
  std::vector<uint32_t> ch, mk;
  for (uint32_t c : h->dirty_list) if (h->pend_reset[c]) { ch.push_back(c); mk.push_back(h->pend_reset[c]); h->pend_reset[c] = 0; }
  h->dirty_list.clear();
  if (!ch.empty()) {
    if (ch.size() > h->reset_cap) {
      if (h->d_reset_ch) { if (dev_sync(h->last_stream)) return SDR_ERR_CUDA; dev_free(h->d_reset_ch); dev_free(h->d_reset_mask); }
      size_t cap = std::max<size_t>(ch.size() * 2, 1024);
      if (dev_alloc((void **)&h->d_reset_ch, cap * 4) || dev_alloc((void **)&h->d_reset_mask, cap * 4)) return SDR_ERR_NOMEM;
      h->reset_cap = cap;
    }
#ifdef SDR_EMU
    /* the host emulation's reset replays the setter side effects only: a slot turn runs here, on the host copy of the state,
     * with the permutation export / import use (the CUDA reset kernel turns the same slots on the device) */
    for (size_t i = 0; i < ch.size(); i++) {
      if ((mk[i] & (SDRK_R_TURN1 | SDRK_R_TURN2)) && !(mk[i] & SDRK_R_NB)) {
        std::vector<float> w(SDR_STATE_WORDS);
        sdrk_launch_gather(h->d_state, h->ch_stride, &ch[i], 1, nullptr, SDR_STATE_WORDS, w.data(), stream);
        rotate_slots(w.data(), (mk[i] & SDRK_R_TURN1) ? 1u : 2u);
        sdrk_launch_scatter(h->d_state, h->ch_stride, &ch[i], 1, w.data(), stream);
      }
      mk[i] &= ~(uint32_t)(SDRK_R_TURN1 | SDRK_R_TURN2);
    }
#endif
    for (size_t o = 0; o < ch.size(); o += 65535) { /* gridDim.y limit */
      uint32_t n = (uint32_t)std::min<size_t>(65535, ch.size() - o);
      if (h2d(h->d_reset_ch + o, ch.data() + o, n * 4, stream) || h2d(h->d_reset_mask + o, mk.data() + o, n * 4, stream)) return SDR_ERR_CUDA;
      /* the staging vectors die at scope exit: the copies above are from pageable memory and complete before return */
      int e = sdrk_launch_reset(h->d_state, h->ch_stride, h->d_reset_ch + o, h->d_reset_mask + o, n, stream);
      if (e) return fail(SDR_ERR_CUDA, "reset kernel launch failed");
      h->launches++;
    }
  }
  return 0;
}

/* fold the per-group profile rows into the per-class sums and clear the device buffer */
int fold_profile(sdr_batch *h) {
  if (!h->d_prof || !h->prof_launches) return 0;
  if (dev_sync(h->last_stream)) return SDR_ERR_CUDA;
  const std::vector<SdrGroup> &groups = (h->prof_of ? h->sub : h->all).groups;
  std::vector<unsigned long long> rows(std::min(groups.size(), h->prof_cap / (SDR_PROF_SLOTS * 8)) * SDR_PROF_SLOTS);
  if (rows.empty()) return 0;
  if (d2h(rows.data(), h->d_prof, rows.size() * 8, h->last_stream) || dev_sync(h->last_stream)) return SDR_ERR_CUDA;
  for (uint32_t g = 0; g < rows.size() / SDR_PROF_SLOTS; g++) {
    int cls = groups[g].cls;
    /* row layout (sdr_kernel.cu pipeline_loop, Probe::flush): [0..13] busy cycles per stage, [14] CTA pipeline cycles, [15] prologue,
     * [16..29] cycles per stage spent waiting for other stages, [30..32] NB sub-phases, [33..35] IN sub-phases */
    for (int w = 0; w < SDR_STAGES; w++) h->prof_busy[cls * SDR_STAGES + w] += rows[(size_t)g * SDR_PROF_SLOTS + w];
    h->prof_total[cls] += rows[(size_t)g * SDR_PROF_SLOTS + 14];
    for (int e = 0; e < 6; e++) h->prof_extra[cls * 8 + e] += rows[(size_t)g * SDR_PROF_SLOTS + 30 + e];
    h->prof_load[cls * (SDR_STAGES + 1) + SDR_STAGES] += rows[(size_t)g * SDR_PROF_SLOTS + 15];
    for (int e = 0; e < SDR_STAGES; e++) h->prof_bar[cls * SDR_STAGES + e] += rows[(size_t)g * SDR_PROF_SLOTS + 16 + e];
    h->prof_groups[cls] += h->prof_launches;
  }
  if (dev_zero(h->d_prof, rows.size() * 8, h->last_stream)) return SDR_ERR_CUDA;
  h->prof_launches = 0;
  return 0;
}

/* A subset call's id list: ids == nullptr stands for every channel (n_ids == n_channels); otherwise 1 <= n_ids, every id below
 * n_channels and none twice. */
int check_ids(sdr_batch *h, const uint32_t *ids, uint32_t n_ids) {
  if (!ids) return n_ids == h->n_ch ? 0 : fail(SDR_ERR_ARG, "channel_ids == NULL needs n_ids == n_channels");
  if (n_ids == 0) return fail(SDR_ERR_ARG, "n_ids == 0");
  uint32_t i = 0;
  for (; i < n_ids && ids[i] < h->n_ch && !h->id_mark[ids[i]]; i++) h->id_mark[ids[i]] = 1;
  for (uint32_t k = 0; k < i; k++) h->id_mark[ids[k]] = 0;
  if (i == n_ids) return 0;
  return fail(SDR_ERR_ARG, ids[i] >= h->n_ch ? "channel id out of range" : "channel id listed twice");
}

bool is_every_channel(const sdr_batch *h, const uint32_t *ids, uint32_t n_ids) {
  if (n_ids != h->n_ch) return false;
  for (uint32_t i = 0; i < n_ids; i++) if (ids[i] != i) return false;
  return true;
}

/* Channels of the call (ids == nullptr: every channel) whose blanker slots are laid out for an earlier block clock get
 * them turned onto the handle's clock, replayed with the setter side effects before the call's launches. */
void queue_turns(sdr_batch *h, const uint32_t *ids, uint32_t n_ids) {
  const uint64_t clk = h->blocks_done;
  for (uint32_t i = 0; i < n_ids; i++) {
    const uint32_t c = ids ? ids[i] : i;
    const uint32_t d = (uint32_t)((clk - std::max(h->plain_at, h->at[c])) % 3);
    if (d) {
      if (!h->pend_reset[c]) h->dirty_list.push_back(c);
      h->pend_reset[c] |= d == 1 ? SDRK_R_TURN1 : SDRK_R_TURN2;
    }
    h->at[c] = clk;
  }
}

int check_plane(const void *p, size_t pitch, int fmt, uint32_t n_blocks, const char *what) {
  if (!p) return fail(SDR_ERR_ARG, std::string(what) + ": null plane");
  if (fmt != SDR_FMT_I16 && fmt != SDR_FMT_F32) return fail(SDR_ERR_ARG, std::string(what) + ": unknown format");
  size_t es = fmt == SDR_FMT_F32 ? 4 : 2;
  if (pitch < (size_t)n_blocks * SDR_BLOCK_SAMPLES) return fail(SDR_ERR_ARG, std::string(what) + ": pitch shorter than the call");
  if ((pitch * es) % 16 != 0 || ((uintptr_t)p) % 16 != 0) return fail(SDR_ERR_ARG, std::string(what) + ": rows must be 16-byte aligned");
  return 0;
}

}  // namespace

extern "C" {

const char *sdr_batch_last_error(void) { return g_err.c_str(); }
const char *sdr_batch_version(void) {
#ifdef SDR_EMU
  return "sdr_batch 0.1 (HOST EMULATION BUILD - tests only)";
#else
  return "sdr_batch 0.1 (sm_100a)";
#endif
}
uint64_t sdr_batch_launch_count(const sdr_batch_t *h) { return h ? h->launches : 0; }

void sdr_batch_destroy(sdr_batch_t *h) {
  if (!h) return;
  dev_select(h->desc.device);
  dev_sync(h->last_stream);
  dev_free(h->d_state); dev_free(h->d_cfg); dev_free(h->all.d_groups); dev_free(h->sub.d_groups); dev_free(h->d_luts); dev_free(h->d_tabs);
  dev_free(h->d_reset_ch); dev_free(h->d_reset_mask); dev_free(h->d_gather); dev_free(h->d_gather_ids); dev_free(h->d_gather_words);
  for (int k = 0; k < 2; k++) {
    dev_free(h->d_in_i[k]); dev_free(h->d_in_q[k]); dev_free(h->d_out[k]); dev_free(h->d_bs[k]);
    dev_event_destroy(h->ev_h2d[k]); dev_event_destroy(h->ev_comp[k]); dev_event_destroy(h->ev_d2h[k]);
  }
  dev_stream_destroy(h->s_h2d); dev_stream_destroy(h->s_comp); dev_stream_destroy(h->s_d2h);
  for (int k = 0; k < SDR_HOST_TICKETS; k++) dev_event_destroy(h->ev_call[k]);
  for (int k = 0; k < SDR_MAX_BUCKETS; k++) { if (h->s_aux[k]) dev_sync(h->s_aux[k]); dev_stream_destroy(h->s_aux[k]); dev_event_destroy(h->ev_join[k]); }
  dev_event_destroy(h->ev_fork);
  dev_free(h->d_prof);
  for (int k = 0; k < SDR_MAX_BUCKETS; k++) dev_free(h->d_raw[k]);
  delete h;
}

int sdr_batch_create(sdr_batch_t **out, const sdr_batch_desc *desc) {
  if (!out || !desc || desc->n_channels == 0) return fail(SDR_ERR_ARG, "create: bad arguments");
  *out = nullptr;
  if (dev_select(desc->device)) return SDR_ERR_CUDA;
  sdr_batch *h = new sdr_batch();
  h->desc = *desc; h->n_ch = desc->n_channels;
  h->ch_stride = ((size_t)h->n_ch + 31) / 32 * 32;
  h->sh.resize(h->n_ch); h->pend_reset.assign(h->n_ch, 0); h->h_cfg.resize(h->n_ch); h->cfg_mark.assign(h->n_ch, 0);
  h->at.assign(h->n_ch, 0); h->own.assign(h->n_ch, 0); h->id_mark.assign(h->n_ch, 0);
  h->plain_at = 0; h->sub_since_plain = false; h->sub_valid = false; h->prof_of = 0;
  h->all.d_groups = h->sub.d_groups = nullptr; h->all.cap = h->sub.cap = 0;
  h->cfg_dirty = h->groups_dirty = true; h->luts_dirty = false; h->cfg_all = true; h->lut_gc_at = 64;
  h->d_state = nullptr; h->d_cfg = nullptr; h->d_luts = nullptr; h->d_tabs = nullptr;
  h->d_reset_ch = h->d_reset_mask = nullptr; h->reset_cap = h->luts_cap = 0;
  h->d_gather = nullptr; h->d_gather_ids = h->d_gather_words = nullptr; h->gather_cap = 0;
  for (int k = 0; k < 2; k++) { h->d_in_i[k] = h->d_in_q[k] = h->d_out[k] = h->d_bs[k] = nullptr; h->ev_h2d[k] = h->ev_comp[k] = h->ev_d2h[k] = nullptr; }
  h->s_h2d = h->s_comp = h->s_d2h = nullptr; h->stage_in_bytes = h->stage_out_bytes = h->stage_bs_bytes = 0; h->host_seq = 0;
  h->host_calls = 0; for (int k = 0; k < SDR_HOST_TICKETS; k++) h->ev_call[k] = nullptr;
  h->blocks_done = 0; h->launches = 0; h->last_stream = nullptr;
  h->d_prof = nullptr; h->prof_cap = 0; h->prof_launches = 0;
  for (int k = 0; k < SDR_MAX_BUCKETS; k++) { h->d_raw[k] = nullptr; h->raw_cap[k] = 0; }
  h->ev_fork = nullptr; for (int k = 0; k < SDR_MAX_BUCKETS; k++) { h->s_aux[k] = nullptr; h->ev_join[k] = nullptr; }
  { const char *e = getenv("SDR_ROLE_PROFILE"); h->prof_on = e && e[0] == '1'; }
  h->prof_busy.assign(2 * SDR_STAGES, 0); h->prof_crit.assign(32, 0); h->prof_bar.assign(2 * SDR_STAGES, 0); h->prof_extra.assign(16, 0); h->prof_load.assign(2 * (SDR_STAGES + 1), 0); h->prof_total.assign(2, 0); h->prof_groups.assign(2, 0);

  SdrTables *t = new SdrTables();
  const uint32_t *ifs[4] = {SDR_TAB_IF_SSB, SDR_TAB_IF_CW, SDR_TAB_IF_WSPR, SDR_TAB_IF_AM};
  const uint32_t *auds[10] = {SDR_TAB_AUDIO_AM, SDR_TAB_AUDIO_CW, SDR_TAB_AUDIO_WSPR, SDR_TAB_AUDIO_2100, SDR_TAB_AUDIO_2300,
                              SDR_TAB_AUDIO_2500, SDR_TAB_AUDIO_2700, SDR_TAB_AUDIO_2900, SDR_TAB_AUDIO_3100, SDR_TAB_AUDIO_3300};
  for (int s = 0; s < 4; s++) for (int i = 0; i < 20; i++) t->if_sets[s][i] = tabf(ifs[s], i);
  for (int s = 0; s < 10; s++) for (int i = 0; i < 20; i++) t->aud_sets[s][i] = tabf(auds[s], i);
  for (int i = 0; i < 20; i++) t->am_image[i] = tabf(SDR_TAB_AM_IMAGE, i);
  for (int i = 0; i < 64; i++) t->hilbert[i] = tabf(SDR_TAB_HILBERT, i);
  { const float k[8] = {1.0f, 1.0f, -1.0f, -1.0f, -0.0f, -0.0f, 0.0f, 0.0f}; memcpy(t->pk_consts, k, sizeof k); }
  memset(t->sine, 0, sizeof t->sine);
  for (int i = 0; i < 257; i++) t->sine[i] = tabf(SDR_TAB_SINE, i);

  int rc = 0;
  do {
    if ((rc = sdrk_setup_device(t->hilbert)) != 0) { rc = fail(SDR_ERR_CUDA, "device setup failed (no sm_100a kernel image or no CUDA device)"); break; }
    if ((rc = dev_alloc((void **)&h->d_state, sizeof(float) * SDR_STATE_WORDS * h->ch_stride)) != 0) break;
    if ((rc = dev_zero(h->d_state, sizeof(float) * SDR_STATE_WORDS * h->ch_stride, nullptr)) != 0) break;
    if ((rc = dev_alloc((void **)&h->d_cfg, sizeof(SdrChanCfg) * h->n_ch)) != 0) break;
    if ((rc = dev_alloc((void **)&h->d_tabs, sizeof(SdrTables))) != 0) break;
    if ((rc = h2d(h->d_tabs, t, sizeof(SdrTables), nullptr)) != 0) break;
    /* power-on values that are not zero: _nb_AvgMag = 10.0 (H:242), _agc_is_active = true (H:230) */
    if (sdrk_launch_fill_word(h->d_state, h->ch_stride, W_NB_AVG, 10.0f, h->n_ch, nullptr)) { rc = fail(SDR_ERR_CUDA, "fill kernel"); break; }
    uint32_t one = 1; float onef; memcpy(&onef, &one, 4);
    if (sdrk_launch_fill_word(h->d_state, h->ch_stride, W_AGC_ACTIVE, onef, h->n_ch, nullptr)) { rc = fail(SDR_ERR_CUDA, "fill kernel"); break; }
    h->launches += 2;
    if ((rc = dev_sync(nullptr)) != 0) break;
  } while (0);
  delete t;
  if (rc) { std::string keep = g_err; sdr_batch_destroy(h); g_err = keep; return rc < 0 ? rc : SDR_ERR_CUDA; }
  for (uint32_t c = 0; c < h->n_ch; c++) { construct(h, c); h->pend_reset[c] = 0; /* fresh state is already zero */ }
  *out = h;
  return SDR_OK;
}

int sdr_batch_set(sdr_batch_t *h, const uint32_t *ids, uint32_t n, uint32_t setter, float a0, float a1, float a2) {
  if (!h) return fail(SDR_ERR_ARG, "null handle");
  if (!ids) n = h->n_ch;
  for (uint32_t i = 0; i < n; i++) {
    uint32_t c = ids ? ids[i] : i;
    if (c >= h->n_ch) return fail(SDR_ERR_ARG, "channel id out of range");
    int rc = apply_one(h, c, setter, a0, a1, a2);
    if (rc) return rc;
    if (h->pend_reset[c]) h->dirty_list.push_back(c);
  }
  return SDR_OK;
}

int sdr_batch_configure(sdr_batch_t *h, const sdr_setter_call *calls, uint32_t n_calls) {
  if (!h || (!calls && n_calls)) return fail(SDR_ERR_ARG, "configure: bad arguments");
  for (uint32_t i = 0; i < n_calls; i++) {
    const sdr_setter_call &k = calls[i];
    int rc;
    if (k.channel == SDR_ALL_CHANNELS) rc = sdr_batch_set(h, nullptr, 0, k.setter, k.a0, k.a1, k.a2);
    else rc = sdr_batch_set(h, &k.channel, 1, k.setter, k.a0, k.a1, k.a2);
    if (rc) return rc;
  }
  return SDR_OK;
}

int sdr_batch_process_device(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                             size_t out_pitch, int out_fmt, uint32_t n_blocks, void *stream) {
  return sdr_batch_process_device_status(h, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, nullptr, stream);
}

int sdr_batch_process_device_status(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                                    size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status, void *stream) {
  return sdr_batch_process_device_subset(h, nullptr, h ? h->n_ch : 0, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks,
                                         block_status, stream);
}

int sdr_batch_process_device_subset(sdr_batch_t *h, const uint32_t *ids, uint32_t n_ids, const void *I, const void *Q, size_t in_pitch,
                                    int in_fmt, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status,
                                    void *stream) {
  if (!h) return fail(SDR_ERR_ARG, "null handle");
  { const int rc = check_ids(h, ids, n_ids); if (rc) return rc; }
  if (ids && is_every_channel(h, ids, n_ids)) ids = nullptr; /* the plain call */
  if (n_blocks == 0) return fail(SDR_ERR_ARG, "n_blocks == 0");
  if ((uintptr_t)block_status % 16 != 0) return fail(SDR_ERR_ARG, "block_status: the record buffer must be 16-byte aligned");
  if (h->desc.max_blocks_per_call && n_blocks > h->desc.max_blocks_per_call) return fail(SDR_ERR_ARG, "n_blocks > max_blocks_per_call");
  if (n_blocks > (1u << 24)) return fail(SDR_ERR_ARG, "n_blocks too large (at most 2^24 blocks per call)");
  int rc;
  if ((rc = check_plane(I, in_pitch, in_fmt, n_blocks, "I")) || (rc = check_plane(Q, in_pitch, in_fmt, n_blocks, "Q")) ||
      (rc = check_plane(audio, out_pitch, out_fmt, n_blocks, "audio")))
    return rc;
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  /* configuration uploads, state resets and the kernels of this call must not overtake work an earlier call queued on
   * another stream (they share the handle's state and tables) */
  if (h->launches && stream != h->last_stream && dev_sync(h->last_stream)) return SDR_ERR_CUDA;
  if (getenv("SDR_MAP_SEARCH")) h->groups_dirty = true; /* tools/map_search.py: plan (and read the placement variables) at every call */
  if (ids || h->sub_since_plain) queue_turns(h, ids, n_ids); /* (nothing lags while only plain calls are made) */
  if ((rc = sync_config(h, stream)) != 0) return rc;
  Grouping &G = ids ? h->sub : h->all;
  if (ids && (!h->sub_valid || h->sub_ids.size() != n_ids || !std::equal(ids, ids + n_ids, h->sub_ids.begin()))) {
    if (h->prof_on && h->prof_of == 1 && fold_profile(h)) return SDR_ERR_CUDA; /* rows are per group: fold before the grouping changes */
    h->sub_valid = false;
    if ((rc = build_groups(h, h->sub, ids, n_ids)) != 0 || (rc = upload_groups(h, h->sub, stream)) != 0) return rc;
    h->sub_ids.assign(ids, ids + n_ids); h->sub_valid = true;
  }
  if (h->prof_on && h->prof_of != (ids ? 1 : 0)) {
    if (fold_profile(h)) return SDR_ERR_CUDA;
    h->prof_of = ids ? 1 : 0;
  }
  SdrLaunch L;
  memset(&L, 0, sizeof L);
  L.in_i = I; L.in_q = Q; L.out = audio; L.in_pitch = in_pitch; L.out_pitch = out_pitch; L.in_fmt = in_fmt; L.out_fmt = out_fmt;
  L.blk0_mod3 = (uint32_t)(h->blocks_done % 3);
  L.flags = h->desc.flags & SDR_BATCH_CONTRACT;
  L.cfg = h->d_cfg; L.state = h->d_state; L.ch_stride = h->ch_stride; L.agc_luts = h->d_luts; L.tabs = h->d_tabs;
  L.bstat = (uint32_t *)block_status; L.bs_stride = n_ids; /* every bucket writes the records of its own channels */
  if (h->prof_on) {
    size_t need = std::max<size_t>(G.groups.size(), 1) * SDR_PROF_SLOTS * 8;
    if (need > h->prof_cap) {
      dev_free(h->d_prof); h->d_prof = nullptr;
      if (dev_alloc((void **)&h->d_prof, need) || dev_zero(h->d_prof, need, stream)) return SDR_ERR_NOMEM;
      h->prof_cap = need;
    }
    h->prof_launches++;
    if (const char *e = getenv("SDR_DIAG_SKIP")) L.diag_skip = (uint32_t)strtoul(e, nullptr, 16); /* time stages in isolation */
  }
  /* one launch per bucket; the first on the caller's stream, the others on streams forked from it and joined back, so
   * that the buckets of a mixed handle share the GPU instead of queueing behind each other */
  const size_t nbk = G.buckets.size();
  if (nbk > 1) {
    if (!h->ev_fork) {
      if (dev_event_create(&h->ev_fork)) return SDR_ERR_CUDA;
      for (int k = 0; k < SDR_MAX_BUCKETS; k++) if (dev_stream_create(&h->s_aux[k]) || dev_event_create(&h->ev_join[k])) return SDR_ERR_CUDA;
    }
    if (dev_event_record(h->ev_fork, stream)) return SDR_ERR_CUDA;
  }
  for (size_t k = 0; k < nbk; k++) {
    const Bucket &b = G.buckets[k];
    void *s = k == 0 ? stream : h->s_aux[k - 1];
    if (k > 0 && dev_stream_wait(s, h->ev_fork)) return SDR_ERR_CUDA;
    L.lay = b.lay; L.groups = G.d_groups + b.first; L.n_groups = b.count;
    L.n_tiles = n_blocks * (uint32_t)b.lay.tpb;
    L.prof = h->prof_on ? h->d_prof + (size_t)b.first * SDR_PROF_SLOTS : nullptr;
    if (getenv("SDR_DEBUG_PLAN")) {
      static int shown = 0;
      const bool two = b.split && !h->prof_on;
      auto show = [&](const SdrLay &y, const char *what) {
        SdrLaunch P = L; P.lay = y;
        fprintf(stderr, "[sdr] %s: class %d feat %u T %d warps %d smem %d B groups %u -> %d CTA(s)/SM; rings nr %d na %d nc %d ni %d hq %d nz %d nz2 %d, input depth %d\n",
                what, y.cls, y.feat, y.T, y.n_warps, y.smem_bytes, b.count, sdrk_occupancy(&P), y.nr, y.na, y.nc, y.ni, y.hq_tiles, y.nz, y.nz2, y.in_depth);
      };
      if (shown++ < 8) {
        if (two) { show(b.lay_main, "launch (chain of a split ALS bucket)"); show(b.lay_als, "launch (ALS post-pass)"); }
        else show(b.lay, "launch");
      }
    }
    if (b.split && !h->prof_on) {
      /* two launches per slice of the call; the scratch plane holds one slice (SDR_ALS_SCRATCH_MB bounds it, 4 GB by default:
       * a slice is then 2 048 blocks of 16 384 channels, long enough that the state reload per slice does not show) */
      const size_t per_block = (size_t)b.count * SDR_BLOCK_SAMPLES * SDR_LANES * sizeof(float);
      const size_t cap = (size_t)std::max(env_int("SDR_ALS_SCRATCH_MB", 4096), 1) << 20;
      const uint32_t slice = (uint32_t)std::min<size_t>(n_blocks, std::max<size_t>(cap / per_block, 16));
      if (h->raw_cap[k] < slice * per_block) {
        if (h->d_raw[k]) { if (dev_sync(h->last_stream)) return SDR_ERR_CUDA; dev_free(h->d_raw[k]); h->d_raw[k] = nullptr; h->raw_cap[k] = 0; }
        if (dev_alloc((void **)&h->d_raw[k], slice * per_block)) return SDR_ERR_NOMEM;
        h->raw_cap[k] = slice * per_block;
      }
      const size_t ies = in_fmt == SDR_FMT_F32 ? 4 : 2, oes = out_fmt == SDR_FMT_F32 ? 4 : 2;
      for (uint32_t b0 = 0; b0 < n_blocks; b0 += slice) {
        const uint32_t nb = std::min(slice, n_blocks - b0);
        SdrLaunch M = L;
        M.in_i = (const char *)I + (size_t)b0 * SDR_BLOCK_SAMPLES * ies; M.in_q = (const char *)Q + (size_t)b0 * SDR_BLOCK_SAMPLES * ies;
        M.out = (char *)audio + (size_t)b0 * SDR_BLOCK_SAMPLES * oes;
        M.blk0_mod3 = (uint32_t)((h->blocks_done + b0) % 3);
        M.raw = h->d_raw[k];
        SdrLaunch A = M;
        A.bstat = nullptr; /* the records come from the chain launch (its AGC stage), the post-pass writes none */
        if (M.bstat) M.bstat += (size_t)b0 * SDR_BS_FIELDS * n_ids;
        M.lay = b.lay_main; M.n_tiles = nb * (uint32_t)b.lay_main.tpb; M.flags |= SDRL_RAW_OUT;
        A.lay = b.lay_als; A.n_tiles = nb * (uint32_t)b.lay_als.tpb;
        A.lay.smem_bytes += env_int("SDR_ALS_PASS_PAD", 0); /* experiment: fewer groups per SM in the post-pass */
        int e = sdrk_launch_pipeline(&M, s);
        if (!e) e = sdrk_launch_als_pass(&A, s);
        if (e) return fail(SDR_ERR_CUDA, "pipeline kernel launch failed (error " + std::to_string(e) + ")");
        h->launches += 2;
      }
    } else {
      int e = sdrk_launch_pipeline(&L, s);
      if (e) return fail(SDR_ERR_CUDA, "pipeline kernel launch failed (error " + std::to_string(e) + ")");
      h->launches++;
    }
    if (k > 0 && (dev_event_record(h->ev_join[k - 1], s) || dev_stream_wait(stream, h->ev_join[k - 1]))) return SDR_ERR_CUDA;
  }
  h->blocks_done += n_blocks;
  if (ids) {
    for (uint32_t i = 0; i < n_ids; i++) { h->at[ids[i]] = h->blocks_done; h->own[ids[i]] += n_blocks; }
    h->sub_since_plain = true;
  } else {
    h->plain_at = h->blocks_done; h->sub_since_plain = false;
  }
  h->last_stream = stream;
  return SDR_OK;
}

int sdr_batch_process(sdr_batch_t *h, const float *I, const float *Q, float *audio, uint32_t n_blocks, void *cuda_stream) {
  const size_t pitch = (size_t)n_blocks * SDR_BLOCK_SAMPLES; /* densely packed float32 rows */
  return sdr_batch_process_device(h, I, Q, pitch, SDR_FMT_F32, audio, pitch, SDR_FMT_F32, n_blocks, cuda_stream);
}

int sdr_batch_wait_host(sdr_batch_t *h) {
  if (!h) return fail(SDR_ERR_ARG, "wait_host: bad arguments");
  if (!h->s_comp) return SDR_OK; /* nothing was ever submitted */
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  if (dev_sync(h->s_d2h) | dev_sync(h->s_comp) | dev_sync(h->s_h2d)) return SDR_ERR_CUDA; /* all three are drained either way */
  return SDR_OK;
}

uint64_t sdr_batch_host_ticket(const sdr_batch_t *h) { return h ? h->host_calls : 0; }

int sdr_batch_wait_host_ticket(sdr_batch_t *h, uint64_t ticket) {
  if (!h) return fail(SDR_ERR_ARG, "wait_host_ticket: bad arguments");
  if (ticket > h->host_calls) return fail(SDR_ERR_ARG, "wait_host_ticket: no such call yet");
  if (ticket == 0 || !h->s_comp) return SDR_OK;
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  /* copy-outs complete in the order of the calls: a ticket whose event has been reused is covered by the oldest one still kept */
  const uint64_t oldest = h->host_calls >= SDR_HOST_TICKETS ? h->host_calls - SDR_HOST_TICKETS + 1 : 1;
  const uint64_t t = ticket < oldest ? oldest : ticket;
  return dev_event_sync(h->ev_call[t % SDR_HOST_TICKETS]) ? SDR_ERR_CUDA : SDR_OK;
}

static int host_call(sdr_batch_t *h, const uint32_t *ids, uint32_t n_ids, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                     void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status, bool streamed);

int sdr_batch_process_host(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                           size_t out_pitch, int out_fmt, uint32_t n_blocks) {
  return sdr_batch_process_host_status(h, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, nullptr);
}

int sdr_batch_process_host_status(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                                  size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status) {
  return sdr_batch_process_host_subset(h, nullptr, h ? h->n_ch : 0, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status);
}

int sdr_batch_process_host_subset(sdr_batch_t *h, const uint32_t *ids, uint32_t n_ids, const void *I, const void *Q, size_t in_pitch,
                                  int in_fmt, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status) {
  const int rc = host_call(h, ids, n_ids, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status, false);
  if (rc) return rc; /* (the streams have been drained) */
  return sdr_batch_wait_host(h);
}

int sdr_batch_submit_host(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                          size_t out_pitch, int out_fmt, uint32_t n_blocks) {
  return sdr_batch_submit_host_status(h, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, nullptr);
}

int sdr_batch_submit_host_status(sdr_batch_t *h, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                                 size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status) {
  return sdr_batch_submit_host_subset(h, nullptr, h ? h->n_ch : 0, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status);
}

int sdr_batch_submit_host_subset(sdr_batch_t *h, const uint32_t *ids, uint32_t n_ids, const void *I, const void *Q, size_t in_pitch,
                                 int in_fmt, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status) {
  return host_call(h, ids, n_ids, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status, true);
}

static int host_call(sdr_batch_t *h, const uint32_t *ids, uint32_t n_ids, const void *I, const void *Q, size_t in_pitch, int in_fmt,
                     void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status, bool streamed) {
  if (!h || !I || !Q || !audio) return fail(SDR_ERR_ARG, "process_host: bad arguments");
  { const int rc = check_ids(h, ids, n_ids); if (rc) return rc; }
  const uint32_t n_rows = n_ids; /* rows of the planes and record columns: one per listed channel */
  if (n_blocks == 0) return fail(SDR_ERR_ARG, "n_blocks == 0");
  if ((uintptr_t)block_status % 16 != 0) return fail(SDR_ERR_ARG, "block_status: the record buffer must be 16-byte aligned");
  if (in_fmt != SDR_FMT_I16 && in_fmt != SDR_FMT_F32) return fail(SDR_ERR_ARG, "process_host: unknown input format");
  if (out_fmt != SDR_FMT_I16 && out_fmt != SDR_FMT_F32) return fail(SDR_ERR_ARG, "process_host: unknown output format");
  const size_t ns = (size_t)n_blocks * SDR_BLOCK_SAMPLES;
  if (in_pitch < ns || out_pitch < ns) return fail(SDR_ERR_ARG, "pitch shorter than the call");
  const size_t ies = in_fmt == SDR_FMT_F32 ? 4 : 2, oes = out_fmt == SDR_FMT_F32 ? 4 : 2;
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  /* chunking along time: ~12 chunks per call, at least 16 blocks each (every chunk is one kernel launch that
   * reloads and saves the per-channel state, so chunks should not be tiny).  A synchronous call wants many chunks: its first
   * copy-in and its last kernel + copy-out are exposed.  A streamed call hides both behind its neighbours and wants the
   * rows of its strided copies long instead: 6 chunks (measured on config 2, streamed / synchronous Msps: 2 chunks 11.5 / 9.0,
   * 4: 12.0 / 10.5, 6: 12.3 / 11.0, 8: 11.9 / 11.1, 12: 12.0 / 11.4, 16: 10.9 / 10.6, 24: 10.6 / 10.5; run r02u). */
  static const uint32_t env_chunks = []() { const char *e = getenv("SDR_HOST_CHUNKS"); int v = e ? atoi(e) : 0; return (uint32_t)(v > 0 ? v : 0); }();
  const uint32_t want_chunks = env_chunks ? env_chunks : (streamed ? 6u : 12u);
  static const uint32_t min_chunk = []() { const char *e = getenv("SDR_HOST_MIN_CHUNK"); int v = e ? atoi(e) : 0; return (uint32_t)(v > 0 ? v : 16); }();
  static const uint32_t ramp = []() { const char *e = getenv("SDR_HOST_RAMP"); int v = e ? atoi(e) : -1; return (uint32_t)(v >= 0 ? v : 0); }();
  uint32_t chunk = (n_blocks + want_chunks - 1) / want_chunks;
  if (chunk < min_chunk) chunk = min_chunk;
  if (chunk > n_blocks) chunk = n_blocks;
  if (h->desc.max_blocks_per_call && chunk > h->desc.max_blocks_per_call) chunk = h->desc.max_blocks_per_call;
  const size_t cs = (size_t)chunk * SDR_BLOCK_SAMPLES;
  const size_t in_bytes = cs * ies * n_rows, out_bytes = cs * oes * n_rows;
  if (!h->s_comp) {
    if (dev_stream_create(&h->s_h2d) || dev_stream_create(&h->s_comp) || dev_stream_create(&h->s_d2h)) return SDR_ERR_CUDA;
    for (int k = 0; k < 2; k++)
      if (dev_event_create(&h->ev_h2d[k]) || dev_event_create(&h->ev_comp[k]) || dev_event_create(&h->ev_d2h[k])) return SDR_ERR_CUDA;
    for (int k = 0; k < SDR_HOST_TICKETS; k++) if (dev_event_create(&h->ev_call[k])) return SDR_ERR_CUDA;
  }
  const size_t bs_bytes = block_status ? (size_t)chunk * SDR_BS_FIELDS * n_rows * 4 : 0;
  if (in_bytes > h->stage_in_bytes || out_bytes > h->stage_out_bytes || bs_bytes > h->stage_bs_bytes) {
    dev_sync(h->last_stream); dev_sync(h->s_h2d); dev_sync(h->s_comp); dev_sync(h->s_d2h);
    const bool grow_in = in_bytes > h->stage_in_bytes, grow_out = out_bytes > h->stage_out_bytes, grow_bs = bs_bytes > h->stage_bs_bytes;
    if (grow_in) h->stage_in_bytes = 0; /* (an allocation that fails below leaves no stale size behind: the next call allocates again) */
    if (grow_out) h->stage_out_bytes = 0;
    if (grow_bs) h->stage_bs_bytes = 0;
    for (int k = 0; k < 2; k++) {
      if (grow_bs) {
        dev_free(h->d_bs[k]); h->d_bs[k] = nullptr;
        if (dev_alloc(&h->d_bs[k], bs_bytes)) return SDR_ERR_NOMEM;
      }
      if (grow_in) {
        dev_free(h->d_in_i[k]); dev_free(h->d_in_q[k]); h->d_in_i[k] = h->d_in_q[k] = nullptr;
        if (dev_alloc(&h->d_in_i[k], in_bytes) || dev_alloc(&h->d_in_q[k], in_bytes)) return SDR_ERR_NOMEM;
      }
      if (grow_out) {
        dev_free(h->d_out[k]); h->d_out[k] = nullptr;
        if (dev_alloc(&h->d_out[k], out_bytes)) return SDR_ERR_NOMEM;
      }
    }
    if (grow_in) h->stage_in_bytes = in_bytes;
    if (grow_out) h->stage_out_bytes = out_bytes;
    if (grow_bs) h->stage_bs_bytes = bs_bytes;
  }
  /* work queued by an earlier process_device call on another stream must finish before the state is touched here */
  if (h->last_stream != h->s_comp && dev_sync(h->last_stream)) return SDR_ERR_CUDA;
  /* Chunk lengths: `chunk` blocks each.  SDR_HOST_RAMP=r (experiment, default off) ramps up from r blocks (doubling) at the
   * start of the call and down again at its end: the first copy-in and the last kernel + copy-out are the only parts of the
   * call nothing overlaps.  Measured: no gain beyond the run-to-run spread of the host link (profiles/README.md). */
  std::vector<uint32_t> sizes;
  {
    std::vector<uint32_t> head;
    uint32_t used = 0;
    for (uint32_t r = ramp; r && r < chunk && used + 2 * r + chunk <= n_blocks; r *= 2) { head.push_back(r); used += 2 * r; }
    uint32_t mid = n_blocks - used;
    sizes = head;
    const uint32_t n_mid = (mid + chunk - 1) / chunk;
    for (uint32_t i = 0; i < n_mid; i++) { const uint32_t a = (uint32_t)((uint64_t)mid * i / n_mid), b = (uint32_t)((uint64_t)mid * (i + 1) / n_mid); sizes.push_back(b - a); }
    for (size_t i = head.size(); i-- > 0;) sizes.push_back(head[i]);
  }
  uint32_t done = 0, k = 0;
  int err = 0;
  /* on any failure the loop stops queueing and the streams are drained before returning: asynchronous copies into the
   * caller's buffers must not outlive the call */
#define SDR_TRY(expr) if ((err = (expr)) != 0) break
  while (done < n_blocks) {
    const uint32_t nb = sizes[k];
    const size_t w_in = (size_t)nb * SDR_BLOCK_SAMPLES * ies, w_out = (size_t)nb * SDR_BLOCK_SAMPLES * oes;
    const int b = (int)(h->host_seq & 1); /* the two staging sets keep alternating from call to call */
    const char *srcI = (const char *)I + (size_t)done * SDR_BLOCK_SAMPLES * ies, *srcQ = (const char *)Q + (size_t)done * SDR_BLOCK_SAMPLES * ies;
    char *dst = (char *)audio + (size_t)done * SDR_BLOCK_SAMPLES * oes;
    /* H2D of chunk k into staging set b: the kernel of chunk k-2 (of this call or, with submit_host, of the call before) must
     * be done with it */
    if (h->host_seq >= 2) { SDR_TRY(dev_stream_wait(h->s_h2d, h->ev_comp[b]) ? SDR_ERR_CUDA : 0); }
    SDR_TRY(h2d_2d(h->d_in_i[b], cs * ies, srcI, in_pitch * ies, w_in, n_rows, h->s_h2d) ? SDR_ERR_CUDA : 0);
    SDR_TRY(h2d_2d(h->d_in_q[b], cs * ies, srcQ, in_pitch * ies, w_in, n_rows, h->s_h2d) ? SDR_ERR_CUDA : 0);
    SDR_TRY(dev_event_record(h->ev_h2d[b], h->s_h2d) ? SDR_ERR_CUDA : 0);
    /* kernel of chunk k: needs its input, and the D2H of chunk k-2 must have drained output set b */
    SDR_TRY(dev_stream_wait(h->s_comp, h->ev_h2d[b]) ? SDR_ERR_CUDA : 0);
    if (h->host_seq >= 2) { SDR_TRY(dev_stream_wait(h->s_comp, h->ev_d2h[b]) ? SDR_ERR_CUDA : 0); }
    int rc = sdr_batch_process_device_subset(h, ids, n_ids, h->d_in_i[b], h->d_in_q[b], cs, in_fmt, h->d_out[b], cs, out_fmt, nb,
                                             block_status ? h->d_bs[b] : nullptr, h->s_comp);
    SDR_TRY(rc);
    SDR_TRY(dev_event_record(h->ev_comp[b], h->s_comp) ? SDR_ERR_CUDA : 0);
    /* D2H of chunk k: audio, then its records (block-major: the chunk's blocks are one contiguous range of the caller's buffer) */
    SDR_TRY(dev_stream_wait(h->s_d2h, h->ev_comp[b]) ? SDR_ERR_CUDA : 0);
    SDR_TRY(d2h_2d(dst, out_pitch * oes, h->d_out[b], cs * oes, w_out, n_rows, h->s_d2h) ? SDR_ERR_CUDA : 0);
    if (block_status) {
      const size_t rec = (size_t)SDR_BS_FIELDS * n_rows; /* words per block */
      SDR_TRY(d2h((uint32_t *)block_status + (size_t)done * rec, h->d_bs[b], (size_t)nb * rec * 4, h->s_d2h) ? SDR_ERR_CUDA : 0);
    }
    SDR_TRY(dev_event_record(h->ev_d2h[b], h->s_d2h) ? SDR_ERR_CUDA : 0);
    done += nb; k++; h->host_seq++;
  }
#undef SDR_TRY
  if (err) { dev_sync(h->s_d2h); dev_sync(h->s_comp); dev_sync(h->s_h2d); return err; }
  /* the call's ticket: its last copy-out is the last thing in the copy-out stream */
  h->host_calls++;
  if (dev_event_record(h->ev_call[h->host_calls % SDR_HOST_TICKETS], h->s_d2h)) return SDR_ERR_CUDA;
  return SDR_OK; /* queued: sdr_batch_wait_host() / sdr_batch_wait_host_ticket() complete it */
}

static int gather_words(sdr_batch_t *h, const uint32_t *ids, uint32_t n, const uint32_t *words, uint32_t nw, std::vector<float> &out) {
  size_t tot = (size_t)n * nw;
  if (tot > h->gather_cap) {
    dev_free(h->d_gather); dev_free(h->d_gather_ids); dev_free(h->d_gather_words);
    h->d_gather = nullptr; h->d_gather_ids = h->d_gather_words = nullptr; h->gather_cap = 0;
    if (dev_alloc((void **)&h->d_gather, tot * 4) || dev_alloc((void **)&h->d_gather_ids, (size_t)n * 4) ||
        dev_alloc((void **)&h->d_gather_words, 64 * 4))
      return SDR_ERR_NOMEM;
    h->gather_cap = tot;
  }
  void *s = h->last_stream;
  if (ids && h2d(h->d_gather_ids, ids, (size_t)n * 4, s)) return SDR_ERR_CUDA;
  if (h2d(h->d_gather_words, words, (size_t)nw * 4, s)) return SDR_ERR_CUDA;
  if (sdrk_launch_gather(h->d_state, h->ch_stride, ids ? h->d_gather_ids : nullptr, n, h->d_gather_words, nw, h->d_gather, s))
    return fail(SDR_ERR_CUDA, "gather kernel launch failed");
  h->launches++;
  out.resize(tot);
  if (d2h(out.data(), h->d_gather, tot * 4, s)) return SDR_ERR_CUDA;
  if (dev_sync(s)) return SDR_ERR_CUDA;
  return 0;
}

int sdr_batch_get_status(sdr_batch_t *h, const uint32_t *ids, uint32_t n, sdr_channel_status *out) {
  if (!h || !out) return fail(SDR_ERR_ARG, "get_status: bad arguments");
  if (n == 0) return SDR_OK;
  for (uint32_t i = 0; i < n; i++) if ((ids ? ids[i] : i) >= h->n_ch) return fail(SDR_ERR_ARG, "channel id out of range");
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  const uint32_t words[8] = {W_AGC_GAIN, W_AGC_ACTIVE, W_AGC_CARRIER, W_SAM_FREQ, W_SAM_LOCKED, W_NB_AVG, W_NB_HIT, W_PH_SSB};
  std::vector<float> v;
  int rc = gather_words(h, ids, n, words, 8, v);
  if (rc) return rc;
  for (uint32_t i = 0; i < n; i++) {
    uint32_t c = ids ? ids[i] : i;
    const Shadow &s = h->sh[c];
    sdr_channel_status &o = out[i];
    memset(&o, 0, sizeof o);
    const float *w = &v[(size_t)i * 8];
    uint32_t u;
    o.tuning_offset = s.freq_shift; o.mode = s.mode; o.audio_filter = s.aud_id; o.muted = s.muted;
    int m = s.mode; /* getBPFlower/upper, C:259-273 */
    if (m == SDR_USB || m == SDR_LSB) { o.bpf_lower = IF_CENTER - BW_SSB / 2.0; o.bpf_upper = IF_CENTER + BW_SSB / 2.0; }
    else if (m == SDR_CW_USB || m == SDR_CW_LSB) { o.bpf_lower = IF_CENTER - BW_CW / 2.0; o.bpf_upper = IF_CENTER + BW_CW / 2.0; }
    else if (m == SDR_AM || m == SDR_SAM) { o.bpf_lower = IF_CENTER - BW_AM / 2.0; o.bpf_upper = IF_CENTER + BW_AM / 2.0; }
    else if (m == SDR_WSPR) { o.bpf_lower = IF_CENTER - BW_WSPR / 2.0; o.bpf_upper = IF_CENTER + -BW_WSPR / 2.0; /* `+-` typo kept, Q11 */ }
    o.agc_gain = w[0]; memcpy(&u, &w[1], 4); o.agc_active = u != 0; o.am_carrier = w[2]; o.sam_frequency = w[3];
    memcpy(&u, &w[4], 4); o.sam_locked = u != 0; o.nb_average = w[5]; memcpy(&u, &w[6], 4); o.nb_detected = u != 0;
    o.agc_enabled = s.agc_on; o.nb_enabled = s.nb_on; o.als_enabled = s.als_on; o.als_notch = s.als_notch; o.als_adaptive = s.als_adapt;
    o.audio_filter_enabled = s.aud_on;
  }
  return SDR_OK;
}

/* ---- checkpoint: a channel's whole carry-over (setter shadow + device state) as one blob */
namespace {
const uint32_t STATE_MAGIC = 0x53445242u; /* "SDRB" */
struct StateHeader { uint32_t magic, version, phase, shadow_bytes; };
size_t state_blob_bytes() { return sizeof(StateHeader) + ((sizeof(Shadow) + 15) / 16) * 16 + sizeof(float) * SDR_STATE_WORDS; }
}  // namespace

size_t sdr_batch_state_bytes(void) { return state_blob_bytes(); }

int sdr_batch_export_state(sdr_batch_t *h, const uint32_t *ids, uint32_t n, void *blobs) {
  if (!h || !blobs) return fail(SDR_ERR_ARG, "export_state: bad arguments");
  if (n == 0) return SDR_OK;
  for (uint32_t i = 0; i < n; i++) if ((ids ? ids[i] : i) >= h->n_ch) return fail(SDR_ERR_ARG, "channel id out of range");
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  int rc = sync_config(h, h->last_stream); /* pending re-initialisations belong to the state being saved */
  if (rc) return rc;
  void *s = h->last_stream;
  float *d_out = nullptr; uint32_t *d_ids = nullptr;
  std::vector<float> words((size_t)n * SDR_STATE_WORDS);
  do {
    if ((rc = dev_alloc((void **)&d_out, words.size() * 4)) != 0) break;
    if (ids) { if ((rc = dev_alloc((void **)&d_ids, (size_t)n * 4)) != 0 || (rc = h2d(d_ids, ids, (size_t)n * 4, s)) != 0) break; }
    if (sdrk_launch_gather(h->d_state, h->ch_stride, d_ids, n, nullptr, SDR_STATE_WORDS, d_out, s)) { rc = fail(SDR_ERR_CUDA, "gather kernel launch failed"); break; }
    h->launches++;
    if ((rc = d2h(words.data(), d_out, words.size() * 4, s)) != 0 || (rc = dev_sync(s)) != 0) break;
  } while (0);
  dev_free(d_out); dev_free(d_ids);
  if (rc) return rc;
  const size_t bb = state_blob_bytes(), so = sizeof(StateHeader), wo = so + ((sizeof(Shadow) + 15) / 16) * 16;
  for (uint32_t i = 0; i < n; i++) {
    char *b = (char *)blobs + (size_t)i * bb;
    memset(b, 0, bb);
    const uint32_t c = ids ? ids[i] : i;
    StateHeader hd = {STATE_MAGIC, 1u, (uint32_t)(std::max(h->plain_at, h->at[c]) % 3), (uint32_t)sizeof(Shadow)}; /* the clock its slots are laid out for */
    memcpy(b, &hd, sizeof hd);
    memcpy(b + so, &h->sh[c], sizeof(Shadow));
    memcpy(b + wo, &words[(size_t)i * SDR_STATE_WORDS], sizeof(float) * SDR_STATE_WORDS);
  }
  return SDR_OK;
}

int sdr_batch_import_state(sdr_batch_t *h, const uint32_t *ids, uint32_t n, const void *blobs) {
  if (!h || !blobs) return fail(SDR_ERR_ARG, "import_state: bad arguments");
  if (n == 0) return SDR_OK;
  const size_t bb = state_blob_bytes(), so = sizeof(StateHeader), wo = so + ((sizeof(Shadow) + 15) / 16) * 16;
  for (uint32_t i = 0; i < n; i++) {
    if ((ids ? ids[i] : i) >= h->n_ch) return fail(SDR_ERR_ARG, "channel id out of range");
    StateHeader hd; memcpy(&hd, (const char *)blobs + (size_t)i * bb, sizeof hd);
    if (hd.magic != STATE_MAGIC || hd.version != 1u || hd.shadow_bytes != sizeof(Shadow) || hd.phase > 2)
      return fail(SDR_ERR_ARG, "import_state: not a state blob of this library version");
  }
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  int rc = sync_config(h, h->last_stream); /* earlier setter calls of the target channels are superseded; flush the others in order */
  if (rc) return rc;
  std::vector<float> words((size_t)n * SDR_STATE_WORDS);
  std::vector<uint32_t> cid(n);
  for (uint32_t i = 0; i < n; i++) {
    const char *b = (const char *)blobs + (size_t)i * bb;
    StateHeader hd; memcpy(&hd, b, sizeof hd);
    const uint32_t c = ids ? ids[i] : i;
    cid[i] = c;
    Shadow sh; memcpy(&sh, b + so, sizeof sh);
    sh.lut_id = lut_for(h, sh.thr, sh.slope, sh.knee); /* table ids are local to a handle */
    h->sh[c] = sh; h->pend_reset[c] = 0; h->at[c] = h->blocks_done; /* (turned onto this handle's clock below) */
    float *w = &words[(size_t)i * SDR_STATE_WORDS];
    memcpy(w, b + wo, sizeof(float) * SDR_STATE_WORDS);
    rotate_slots(w, (uint32_t)((h->blocks_done % 3) + 3 - hd.phase));
  }
  h->cfg_dirty = true; h->groups_dirty = true; h->cfg_all = true; /* (the shadows were written directly) */
  void *s = h->last_stream;
  float *d_in = nullptr; uint32_t *d_ids = nullptr;
  do {
    if ((rc = dev_alloc((void **)&d_in, words.size() * 4)) != 0 || (rc = dev_alloc((void **)&d_ids, (size_t)n * 4)) != 0) break;
    if ((rc = h2d(d_in, words.data(), words.size() * 4, s)) != 0 || (rc = h2d(d_ids, cid.data(), (size_t)n * 4, s)) != 0) break;
    if (sdrk_launch_scatter(h->d_state, h->ch_stride, d_ids, n, d_in, s)) { rc = fail(SDR_ERR_CUDA, "scatter kernel launch failed"); break; }
    h->launches++;
    rc = dev_sync(s); /* the staging vectors and device buffers die here */
  } while (0);
  dev_free(d_in); dev_free(d_ids);
  return rc;
}

int sdr_batch_get_role_profile(sdr_batch_t *h, uint64_t *busy28, uint64_t *total2, uint64_t *groups2) {
  if (!h || !busy28 || !total2 || !groups2) return fail(SDR_ERR_ARG, "get_role_profile: bad arguments");
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  if (fold_profile(h)) return SDR_ERR_CUDA;
  for (int i = 0; i < 2 * SDR_STAGES; i++) busy28[i] = h->prof_busy[i];
  for (int i = 0; i < 2; i++) { total2[i] = h->prof_total[i]; groups2[i] = h->prof_groups[i]; }
  if (getenv("SDR_ROLE_PROFILE_NB"))
    for (int cls = 0; cls < 2; cls++)
      if (h->prof_groups[cls]) {
        fprintf(stderr, "[sdr] class %d: cycles per CTA launch: prologue %.0f, pipeline %.0f; share of it each stage spent waiting for other stages:", cls,
                (double)h->prof_load[cls * (SDR_STAGES + 1) + SDR_STAGES] / h->prof_groups[cls], (double)h->prof_total[cls] / h->prof_groups[cls]);
        for (int w = 0; w < SDR_STAGES; w++) fprintf(stderr, " %.3f", (double)h->prof_bar[cls * SDR_STAGES + w] / (double)std::max<uint64_t>(h->prof_total[cls], 1));
        fprintf(stderr, "\n");
      }
  if (getenv("SDR_ROLE_PROFILE_NB") && h->prof_total[0])
    fprintf(stderr, "[sdr] sub-phase share of CTA time: nb.wait %.3f nb.scan %.3f nb.edge+request %.3f | in.wait %.3f in.scale+ring %.3f (unused %.3f)\n",
            (double)h->prof_extra[0] / h->prof_total[0], (double)h->prof_extra[1] / h->prof_total[0], (double)h->prof_extra[2] / h->prof_total[0],
            (double)h->prof_extra[3] / h->prof_total[0], (double)h->prof_extra[4] / h->prof_total[0], (double)h->prof_extra[5] / h->prof_total[0]);
  return SDR_OK;
}

int sdr_batch_get_agc_lookup(sdr_batch_t *h, uint32_t channel, float *out129) {
  if (!h || !out129 || channel >= h->n_ch) return fail(SDR_ERR_ARG, "get_agc_lookup: bad arguments");
  memcpy(out129, &h->luts[(size_t)h->sh[channel].lut_id * SDR_AGC_LUT_STRIDE], 129 * sizeof(float));
  return SDR_OK;
}

int sdr_batch_peek_state(sdr_batch_t *h, uint32_t channel, uint32_t word, float *out) {
  if (!h || !out || channel >= h->n_ch || word >= SDR_STATE_WORDS) return fail(SDR_ERR_ARG, "peek_state: bad arguments");
  if (dev_select(h->desc.device)) return SDR_ERR_CUDA;
  std::vector<float> v;
  int rc = gather_words(h, &channel, 1, &word, 1, v);
  if (rc) return rc;
  *out = v[0];
  return SDR_OK;
}

}  // extern "C"
