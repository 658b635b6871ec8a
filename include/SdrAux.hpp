/* include/SdrAux.hpp -- host C++ mirrors of the two blocks in front of the receiver, over the C ABI of sdr_aux.h.
 *
 *   sdr::PreProcessorBatch  <-  class AudioSDRpreProcessor  (AudioSDRpreProcessor.h:49-73)
 *   sdr::IQGeneratorBatch   <-  class AudioIQgenerator      (AudioIQgenerator.h:49-107)
 *   sdr::GrabberBatch       <-  class AudioGrabberComplex256 (AudioGrabberComplex256.h:46-64)
 *
 * Every public method of the reference keeps its name and argument meaning with a channel selector in front
 * (sdr::Channels from SdrBatch.hpp: one id, a vector of ids, or sdr::all); update() becomes process() over int16 planes.
 * process(ids, ...) advances only the listed channels, on compact planes (row i = channel ids[i]); export_state /
 * import_state move channels' whole state as opaque blobs of state_bytes() bytes each (sdr_aux.h).
 * Header only; link against audiosdr_b200/libsdr_aux.so.  Errors of the C ABI become std::runtime_error.
 */
#ifndef SDR_AUX_HPP
#define SDR_AUX_HPP
#include <stdexcept>
#include <string>
#include <vector>

#include "SdrBatch.hpp"
#include "sdr_aux.h"

namespace sdr {

class PreProcessorBatch {
 public:
  explicit PreProcessorBatch(uint32_t n_channels, int device = 0) : h_(nullptr) { check(sdr_preproc_create(&h_, n_channels, device), "sdr_preproc_create"); }
  ~PreProcessorBatch() { sdr_preproc_destroy(h_); }
  PreProcessorBatch(const PreProcessorBatch &) = delete;
  PreProcessorBatch &operator=(const PreProcessorBatch &) = delete;
  /* AudioSDRpreProcessor.h:54-59 */
  void startAutoI2SerrorDetection(Channels c = all) { set(c, SDR_PP_startAutoI2SerrorDetection, 0); }
  void stopAutoI2SerrorDetection(Channels c = all) { set(c, SDR_PP_stopAutoI2SerrorDetection, 0); }
  bool getAutoI2SerrorDetectionStatus(uint32_t c) { return status(c).auto_detect != 0; }
  void setI2SerrorCompensation(Channels c, int correction) { set(c, SDR_PP_setI2SerrorCompensation, correction); }
  int16_t getI2SerrorCompensation(uint32_t c) { return (int16_t)status(c).correction; }
  void swapIQ(Channels c, bool swap) { set(c, SDR_PP_swapIQ, swap ? 1 : 0); }
  sdr_preproc_status status(uint32_t c) {
    sdr_preproc_status s;
    check(sdr_preproc_get_status(h_, &c, 1, &s), "sdr_preproc_get_status");
    return s;
  }
  /* AudioSDRpreProcessor::update() for every channel, n_blocks blocks each (AudioSDRpreProcessor.cpp:46-138); device planes */
  void process(const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
               void *cuda_stream = nullptr) {
    check(sdr_preproc_process_device(h_, I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks, cuda_stream), "sdr_preproc_process_device");
  }
  void process_host(const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks) {
    check(sdr_preproc_process_host(h_, I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks), "sdr_preproc_process_host");
  }
  /* the listed channels only; every other channel skips the call untouched */
  void process(const std::vector<uint32_t> &ids, const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out, int16_t *Q_out,
               size_t out_pitch, uint32_t n_blocks, void *cuda_stream = nullptr) {
    check(sdr_preproc_process_device_subset(h_, ids.data(), (uint32_t)ids.size(), I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks, cuda_stream),
          "sdr_preproc_process_device_subset");
  }
  void process_host(const std::vector<uint32_t> &ids, const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out, int16_t *Q_out,
                    size_t out_pitch, uint32_t n_blocks) {
    check(sdr_preproc_process_host_subset(h_, ids.data(), (uint32_t)ids.size(), I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks),
          "sdr_preproc_process_host_subset");
  }
  static size_t state_bytes() { return sdr_preproc_state_bytes(); }
  std::vector<uint8_t> export_state(const std::vector<uint32_t> &ids) {
    std::vector<uint8_t> b(ids.size() * state_bytes());
    check(sdr_preproc_export_state(h_, ids.data(), (uint32_t)ids.size(), b.data()), "sdr_preproc_export_state");
    return b;
  }
  void import_state(const std::vector<uint32_t> &ids, const std::vector<uint8_t> &blobs) {
    if (blobs.size() != ids.size() * state_bytes()) throw std::runtime_error("import_state: one blob per channel");
    check(sdr_preproc_import_state(h_, ids.data(), (uint32_t)ids.size(), blobs.data()), "sdr_preproc_import_state");
  }
  sdr_preproc_t *handle() { return h_; }

 private:
  void set(const Channels &c, uint32_t setter, int32_t arg) { check(sdr_preproc_set(h_, c.ids, c.n, setter, arg), "sdr_preproc_set"); }
  static void check(int rc, const char *what) {
    if (rc != SDR_AUX_OK) throw std::runtime_error(std::string(what) + ": " + sdr_aux_last_error());
  }
  sdr_preproc_t *h_;
};

class IQGeneratorBatch {
 public:
  explicit IQGeneratorBatch(uint32_t n_channels, int device = 0) : h_(nullptr) { check(sdr_iqgen_create(&h_, n_channels, device), "sdr_iqgen_create"); }
  ~IQGeneratorBatch() { sdr_iqgen_destroy(h_); }
  IQGeneratorBatch(const IQGeneratorBatch &) = delete;
  IQGeneratorBatch &operator=(const IQGeneratorBatch &) = delete;
  /* AudioIQgenerator.h:56-60 */
  void setGainBalance(Channels c, float balance) { check(sdr_iqgen_set_gain_balance(h_, c.ids, c.n, balance), "sdr_iqgen_set_gain_balance"); }
  /* AudioIQgenerator::update() for every channel, n_blocks blocks each (AudioIQgenerator.cpp:33-87); device planes */
  void process(const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks, void *cuda_stream = nullptr) {
    check(sdr_iqgen_process_device(h_, X, in_pitch, I_out, Q_out, out_pitch, n_blocks, cuda_stream), "sdr_iqgen_process_device");
  }
  void process_host(const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks) {
    check(sdr_iqgen_process_host(h_, X, in_pitch, I_out, Q_out, out_pitch, n_blocks), "sdr_iqgen_process_host");
  }
  void process(const std::vector<uint32_t> &ids, const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch,
               uint32_t n_blocks, void *cuda_stream = nullptr) {
    check(sdr_iqgen_process_device_subset(h_, ids.data(), (uint32_t)ids.size(), X, in_pitch, I_out, Q_out, out_pitch, n_blocks, cuda_stream),
          "sdr_iqgen_process_device_subset");
  }
  void process_host(const std::vector<uint32_t> &ids, const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch,
                    uint32_t n_blocks) {
    check(sdr_iqgen_process_host_subset(h_, ids.data(), (uint32_t)ids.size(), X, in_pitch, I_out, Q_out, out_pitch, n_blocks),
          "sdr_iqgen_process_host_subset");
  }
  static size_t state_bytes() { return sdr_iqgen_state_bytes(); }
  std::vector<uint8_t> export_state(const std::vector<uint32_t> &ids) {
    std::vector<uint8_t> b(ids.size() * state_bytes());
    check(sdr_iqgen_export_state(h_, ids.data(), (uint32_t)ids.size(), b.data()), "sdr_iqgen_export_state");
    return b;
  }
  void import_state(const std::vector<uint32_t> &ids, const std::vector<uint8_t> &blobs) {
    if (blobs.size() != ids.size() * state_bytes()) throw std::runtime_error("import_state: one blob per channel");
    check(sdr_iqgen_import_state(h_, ids.data(), (uint32_t)ids.size(), blobs.data()), "sdr_iqgen_import_state");
  }
  sdr_iqgen_t *handle() { return h_; }

 private:
  static void check(int rc, const char *what) {
    if (rc != SDR_AUX_OK) throw std::runtime_error(std::string(what) + ": " + sdr_aux_last_error());
  }
  sdr_iqgen_t *h_;
};

/* AudioGrabberComplex256 (AudioGrabberComplex256.h:46-64) for n channels */
class GrabberBatch {
 public:
  explicit GrabberBatch(uint32_t n_channels, int device = 0) : h_(nullptr), n_channels_(n_channels) {
    check(sdr_grabber_create(&h_, n_channels, device), "sdr_grabber_create");
  }
  ~GrabberBatch() { sdr_grabber_destroy(h_); }
  GrabberBatch(const GrabberBatch &) = delete;
  GrabberBatch &operator=(const GrabberBatch &) = delete;
  /* update() for every channel, n_blocks blocks each; device planes */
  void process(const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, void *cuda_stream = nullptr) {
    check(sdr_grabber_process_device(h_, I, Q, pitch, n_blocks, cuda_stream), "sdr_grabber_process_device");
  }
  void process(const std::vector<uint32_t> &ids, const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, void *cuda_stream = nullptr) {
    check(sdr_grabber_process_device_subset(h_, ids.data(), (uint32_t)ids.size(), I, Q, pitch, n_blocks, cuda_stream), "sdr_grabber_process_device_subset");
  }
  /* ... also every snapshot the call publishes and/or its power spectrum (device [rows][(n_blocks+1)/2][512] int16 and
   * [rows][(n_blocks+1)/2][256] float, either may be null) and the slots written per row (host, rows entries, may be null);
   * sdr_grabber_process_device_snapshots */
  void process(const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, int16_t *snapshots, float *power, uint32_t *counts,
               void *cuda_stream = nullptr) {
    check(sdr_grabber_process_device_snapshots(h_, nullptr, n_channels_, I, Q, pitch, n_blocks, snapshots, power, counts, cuda_stream),
          "sdr_grabber_process_device_snapshots");
  }
  void process(const std::vector<uint32_t> &ids, const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, int16_t *snapshots,
               float *power, uint32_t *counts, void *cuda_stream = nullptr) {
    check(sdr_grabber_process_device_snapshots(h_, ids.data(), (uint32_t)ids.size(), I, Q, pitch, n_blocks, snapshots, power, counts, cuda_stream),
          "sdr_grabber_process_device_snapshots");
  }
  static size_t state_bytes() { return sdr_grabber_state_bytes(); }
  std::vector<uint8_t> export_state(const std::vector<uint32_t> &ids) {
    std::vector<uint8_t> b(ids.size() * state_bytes());
    check(sdr_grabber_export_state(h_, ids.data(), (uint32_t)ids.size(), b.data()), "sdr_grabber_export_state");
    return b;
  }
  void import_state(const std::vector<uint32_t> &ids, const std::vector<uint8_t> &blobs) {
    if (blobs.size() != ids.size() * state_bytes()) throw std::runtime_error("import_state: one blob per channel");
    check(sdr_grabber_import_state(h_, ids.data(), (uint32_t)ids.size(), blobs.data()), "sdr_grabber_import_state");
  }
  bool newDataAvailable(uint32_t c) { const int r = sdr_grabber_new_data_available(h_, c); if (r < 0) check(r, "sdr_grabber_new_data_available"); return r != 0; }
  /* grab(destination) of one channel: 512 int16 to host memory; false (destination untouched) before the first complete pair */
  bool grab(uint32_t c, int16_t *destination) { const int r = sdr_grabber_grab(h_, &c, 1, destination); if (r < 0) check(r, "sdr_grabber_grab"); return r > 0; }
  /* spectrum tap: power[256] of the 256-point FFT of channel c's snapshot (natural bin order); false before the first complete pair */
  bool spectrum(uint32_t c, float *power) { const int r = sdr_grabber_spectrum(h_, &c, 1, power); if (r < 0) check(r, "sdr_grabber_spectrum"); return r > 0; }

 private:
  static void check(int rc, const char *what) {
    if (rc != SDR_AUX_OK) throw std::runtime_error(std::string(what) + ": " + sdr_aux_last_error());
  }
  sdr_grabber_t *h_;
  uint32_t n_channels_;
};

}  // namespace sdr
#endif
