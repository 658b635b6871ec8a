/* include/SdrBatch.hpp -- host C++ mirror of the reference class's interface, over the C ABI of sdr_batch.h.
 *
 * The reference is one C++ object per receiver (`class AudioSDR : public AudioStream`, AudioSDR.h:75-156) whose
 * setters are called from the sketch and whose update() runs in the audio ISR.  `SdrBatch` is N such receivers
 * on one GPU: every public method of the reference keeps its NAME, ARGUMENT MEANING and ERROR BEHAVIOUR (the
 * reference's setters never fail; values outside its enumerations are rejected here instead of leaving a
 * channel without a demodulator), with a channel selector in front:
 *
 *     reference                          batch
 *     SDR.setDemodMode(USBmode);         sdr.setDemodMode(ch, SDR_USB);          // one channel
 *     SDR.enableAGC();                   sdr.enableAGC();                        // every channel
 *     SDR.setAGCmode(AGCmedium);         sdr.setAGCmode(sdr::all, SDR_AGC_MEDIUM);
 *     (audio ISR) SDR.update();          sdr.process(I, Q, audio, n_blocks);     // all channels, n_blocks blocks each
 *     SDR.getSAMfrequency();             sdr.status(ch).sam_frequency;
 *
 * Header only; link against audiosdr_b200/libsdr_batch.so.  Errors of the C ABI become std::runtime_error.
 */
#ifndef SDR_BATCH_HPP
#define SDR_BATCH_HPP
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "sdr_batch.h"

namespace sdr {

/* channel selector: one channel, a list, or all of them */
struct Channels {
  const uint32_t *ids;
  uint32_t n;
  uint32_t one;
  bool every; /* all channels of the handle (an EMPTY list selects nothing: `every` is what tells the two apart) */
  Channels() : ids(nullptr), n(0), one(0), every(true) {}                                    /* all channels */
  Channels(uint32_t c) : ids(&one), n(1), one(c), every(false) {}                            /* NOLINT: implicit on purpose */
  Channels(int c) : ids(&one), n(1), one((uint32_t)c), every(false) {}                       /* NOLINT */
  Channels(const std::vector<uint32_t> &v) : ids(v.data()), n((uint32_t)v.size()), one(0), every(false) {} /* NOLINT */
  Channels(const Channels &o) : ids(o.ids == &o.one ? &one : o.ids), n(o.n), one(o.one), every(o.every) {}
};
static const Channels all;

class SdrBatch {
 public:
  /* AudioSDR::AudioSDR() -> init() for every channel (AudioSDR.h:77-79, AudioSDR.cpp:174-185) */
  explicit SdrBatch(uint32_t n_channels, int device = 0, uint32_t max_blocks_per_call = 0, uint32_t flags = 0) : h_(nullptr), n_(n_channels) {
    sdr_batch_desc d = {n_channels, device, max_blocks_per_call, flags};
    check(sdr_batch_create(&h_, &d), "sdr_batch_create");
  }
  ~SdrBatch() { sdr_batch_destroy(h_); }
  SdrBatch(const SdrBatch &) = delete;
  SdrBatch &operator=(const SdrBatch &) = delete;
  uint32_t channels() const { return n_; }

  /* --- general (AudioSDR.h:88-97) */
  void init(Channels c = all) { set(c, SDR_SET_init); }
  void setMute(Channels c, bool m) { set(c, SDR_SET_setMute, m ? 1.f : 0.f); }
  void setInputGain(Channels c, float g) { set(c, SDR_SET_setInputGain, g); }
  void setIQgainBalance(Channels c, float b) { set(c, SDR_SET_setIQgainBalance, b); }
  /* returns the tuning offset like the reference does (AudioSDR.cpp:220-221) */
  float setDemodMode(Channels c, int mode) {
    set(c, SDR_SET_setDemodMode, (float)mode);
    static const float off[7] = {8390.f, 5390.f, 7390.f, 6390.f, 6890.f, 6890.f, 5390.f};
    return off[mode];
  }
  int16_t getDemodMode(uint32_t c) { return (int16_t)status(c).mode; }
  float getBPFlower(uint32_t c) { return status(c).bpf_lower; }
  float getBPFupper(uint32_t c) { return status(c).bpf_upper; }
  float getTuningOffset(uint32_t c) { return status(c).tuning_offset; }
  bool getMute(uint32_t c) { return status(c).muted != 0; }
  /* --- audio output filters (AudioSDR.h:100-104) */
  void enableAudioFilter(Channels c = all) { set(c, SDR_SET_enableAudioFilter); }
  void disableAudioFilter(Channels c = all) { set(c, SDR_SET_disableAudioFilter); }
  int getAudioFilter(uint32_t c) { return status(c).audio_filter; }
  void setOutputGain(Channels c, float g) { set(c, SDR_SET_setOutputGain, g); }
  void setAudioFilter(Channels c, int f) { set(c, SDR_SET_setAudioFilter, (float)f); }
  /* --- ALS notch / peak filter (AudioSDR.h:107-117) */
  void enableALSfilter(Channels c = all) { set(c, SDR_SET_enableALSfilter); }
  void disableALSfilter(Channels c = all) { set(c, SDR_SET_disableALSfilter); }
  void setALSfilterNotch(Channels c = all) { set(c, SDR_SET_setALSfilterNotch); }
  void setALSfilterPeak(Channels c = all) { set(c, SDR_SET_setALSfilterPeak); }
  void setALSfilterAdaptive(Channels c = all) { set(c, SDR_SET_setALSfilterAdaptive); }
  void setALSfilterStatic(Channels c = all) { set(c, SDR_SET_setALSfilterStatic); }
  void setALSfilterParams(Channels c, unsigned m, float lambda, float delay) { set(c, SDR_SET_setALSfilterParams, (float)m, lambda, delay); }
  bool ALSfilterIsEnabled(uint32_t c) { return status(c).als_enabled != 0; }
  bool ALSfilterIsNotch(uint32_t c) { return status(c).als_notch != 0; }
  bool ALSfilterIsPeak(uint32_t c) { return status(c).als_notch == 0; }
  bool ALSfilterIsAdaptive(uint32_t c) { return status(c).als_adaptive != 0; }
  /* --- AGC (AudioSDR.h:120-144) */
  void enableAGC(Channels c = all) { set(c, SDR_SET_enableAGC); }
  void disableAGC(Channels c = all) { set(c, SDR_SET_disableAGC); }
  bool AGCisEnabled(uint32_t c) { return status(c).agc_enabled != 0; }
  bool AGCisActive(uint32_t c) { return status(c).agc_active != 0; }
  void setAGCthreshold(Channels c, float v) { set(c, SDR_SET_setAGCthreshold, v); }
  void setAGCslope(Channels c, float v) { set(c, SDR_SET_setAGCslope, v); }
  void setAGCmode(Channels c, int16_t m) { set(c, SDR_SET_setAGCmode, (float)m); }
  void setAGCkneeWidth(Channels c, float v) { set(c, SDR_SET_setAGCkneeWidth, v); }
  void setAGCattackTime(Channels c, float ms) { set(c, SDR_SET_setAGCattackTime, ms); }
  void setAGCreleaseTime(Channels c, float ms) { set(c, SDR_SET_setAGCreleaseTime, ms); }
  void setAGChangTime(Channels c, float ms) { set(c, SDR_SET_setAGChangTime, ms); }
  void setAGCstaticGain(Channels c, float g) { set(c, SDR_SET_setAGCstaticGain, g); }
  float getAGClookup(uint32_t c, int i) {
    float lut[129];
    check(sdr_batch_get_agc_lookup(h_, c, lut), "sdr_batch_get_agc_lookup");
    return lut[i];
  }
  float getAMcarrierLevel(uint32_t c) { return status(c).am_carrier; }
  /* --- impulse noise blanker (AudioSDR.h:147-152) */
  void enableNoiseBlanker(Channels c = all) { set(c, SDR_SET_enableNoiseBlanker); }
  void disableNoiseBlanker(Channels c = all) { set(c, SDR_SET_disableNoiseBlanker); }
  void setNoiseBlankerThreshold(Channels c, float ratio) { set(c, SDR_SET_setNoiseBlankerThreshold, ratio); }
  void setNoiseBlankerThresholdDb(Channels c, float db) { set(c, SDR_SET_setNoiseBlankerThresholdDb, db); }
  bool NoiseBlankerisEnabled(uint32_t c) { return status(c).nb_enabled != 0; }
  bool NoiseBlankerDetection(uint32_t c) { return status(c).nb_detected != 0; }
  /* --- synchronous AM detector (AudioSDR.h:155-156) */
  float getSAMfrequency(uint32_t c) { return status(c).sam_frequency; }
  bool getSAMphaseLockStatus(uint32_t c) { return status(c).sam_locked != 0; }

  sdr_channel_status status(uint32_t c) {
    sdr_channel_status s;
    check(sdr_batch_get_status(h_, &c, 1, &s), "sdr_batch_get_status");
    return s;
  }
  /* --- AudioSDR::update() for every channel, n_blocks blocks each (AudioSDR.cpp:39-168).  Device planes. */
  void process(const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt,
               uint32_t n_blocks, void *cuda_stream = nullptr) {
    check(sdr_batch_process_device(h_, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, cuda_stream), "sdr_batch_process_device");
  }
  /* ... host planes (copies in, runs, copies out) */
  void process_host(const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt,
                    uint32_t n_blocks) {
    check(sdr_batch_process_host(h_, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks), "sdr_batch_process_host");
  }
  /* ... the same as a stream of calls: submit_host() queues and returns, wait_host() completes everything queued */
  void submit_host(const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt,
                   uint32_t n_blocks) {
    check(sdr_batch_submit_host(h_, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks), "sdr_batch_submit_host");
  }
  /* ... each of the three with per-block status records: the dynamic getters after every block of the call, block-major
   * [n_blocks][SDR_BS_FIELDS][channels] 32-bit words (sdr_batch.h, SDR_BS_*), 16-byte aligned; device memory for process(),
   * host memory for the host forms (they land with the call's audio).  nullptr = the overload without records. */
  void process(const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt,
               uint32_t n_blocks, void *block_status, void *cuda_stream) {
    check(sdr_batch_process_device_status(h_, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status, cuda_stream),
          "sdr_batch_process_device_status");
  }
  void process_host(const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt,
                    uint32_t n_blocks, void *block_status) {
    check(sdr_batch_process_host_status(h_, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status), "sdr_batch_process_host_status");
  }
  void submit_host(const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio, size_t out_pitch, int out_fmt,
                   uint32_t n_blocks, void *block_status) {
    check(sdr_batch_submit_host_status(h_, I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt, n_blocks, block_status), "sdr_batch_submit_host_status");
  }
  /* ... on the channels `ids` only (sdr_batch_process_*_subset): row i of the planes and record column i belong to ids[i];
   * every other channel skips the call untouched, as update() does without input (AudioSDR.cpp:48-56) */
  void process(const std::vector<uint32_t> &ids, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
               size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status = nullptr, void *cuda_stream = nullptr) {
    check(sdr_batch_process_device_subset(h_, ids.data(), (uint32_t)ids.size(), I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt,
                                          n_blocks, block_status, cuda_stream), "sdr_batch_process_device_subset");
  }
  void process_host(const std::vector<uint32_t> &ids, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                    size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status = nullptr) {
    check(sdr_batch_process_host_subset(h_, ids.data(), (uint32_t)ids.size(), I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt,
                                        n_blocks, block_status), "sdr_batch_process_host_subset");
  }
  void submit_host(const std::vector<uint32_t> &ids, const void *I, const void *Q, size_t in_pitch, int in_fmt, void *audio,
                   size_t out_pitch, int out_fmt, uint32_t n_blocks, void *block_status = nullptr) {
    check(sdr_batch_submit_host_subset(h_, ids.data(), (uint32_t)ids.size(), I, Q, in_pitch, in_fmt, audio, out_pitch, out_fmt,
                                       n_blocks, block_status), "sdr_batch_submit_host_subset");
  }
  void wait_host() { check(sdr_batch_wait_host(h_), "sdr_batch_wait_host"); }
  uint64_t host_ticket() const { return sdr_batch_host_ticket(h_); } /* names the call submitted last */
  void wait_host(uint64_t ticket) { check(sdr_batch_wait_host_ticket(h_, ticket), "sdr_batch_wait_host_ticket"); }
  sdr_batch_t *handle() { return h_; }

 private:
  void set(const Channels &c, uint32_t setter, float a0 = 0.f, float a1 = 0.f, float a2 = 0.f) {
    if (!c.every && c.n == 0) return; /* an empty selection: nothing to do (the C call reads ids == NULL as "all channels") */
    check(sdr_batch_set(h_, c.every ? nullptr : c.ids, c.n, setter, a0, a1, a2), "sdr_batch_set");
  }
  static void check(int rc, const char *what) {
    if (rc != SDR_OK) throw std::runtime_error(std::string(what) + ": " + sdr_batch_last_error());
  }
  sdr_batch_t *h_;
  uint32_t n_;
};

}  // namespace sdr
#endif
