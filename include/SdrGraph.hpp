/* include/SdrGraph.hpp -- host C++ wrapper of the streamed receiver graph, over the C ABI of sdr_graph.h.
 *
 *     sdr::SdrBatch rx(n);  sdr::PreProcessorBatch pp(n);  sdr::GrabberBatch gr(n);
 *     sdr::SdrGraph graph(rx, &pp, nullptr, &gr);              // I2S in -> pre-processor -> receiver, grabber on the I/Q
 *     uint64_t t = graph.submit_host(I, Q, pitch, audio, pitch, SDR_FMT_I16, n_blocks, outputs);
 *     ...                                                      // submit the next call, then
 *     graph.wait_host(t);                                      // audio, records, spectra of call t have landed
 *
 * The graph does not own the member objects: it must be destroyed before them.  Header only; link against
 * audiosdr_b200/libsdr_graph.so (which finds libsdr_batch.so and libsdr_aux.so beside it).  Errors of the C ABI become
 * std::runtime_error.
 */
#ifndef SDR_GRAPH_HPP
#define SDR_GRAPH_HPP
#include <stdexcept>
#include <string>
#include <vector>

#include "SdrAux.hpp"
#include "SdrBatch.hpp"
#include "sdr_graph.h"

namespace sdr {

class SdrGraph {
 public:
  /* at most one of pp / gen (the front); grabber optional */
  SdrGraph(SdrBatch &rx, PreProcessorBatch *pp = nullptr, IQGeneratorBatch *gen = nullptr, GrabberBatch *grabber = nullptr) : g_(nullptr), n_(rx.channels()) {
    const sdr_graph_desc d = {rx.handle(), pp ? pp->handle() : nullptr, gen ? gen->handle() : nullptr, grabber ? grabber->handle() : nullptr};
    check(sdr_graph_create(&g_, &d), "sdr_graph_create");
  }
  ~SdrGraph() { sdr_graph_destroy(g_); }
  SdrGraph(const SdrGraph &) = delete;
  SdrGraph &operator=(const SdrGraph &) = delete;

  /* every channel: host int16 planes (Q == nullptr with the I/Q generator front), returns the call's ticket */
  uint64_t submit_host(const int16_t *I_or_X, const int16_t *Q, size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                       const sdr_graph_outputs *o = nullptr) {
    check(sdr_graph_submit_host(g_, nullptr, n_, I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o), "sdr_graph_submit_host");
    return sdr_graph_host_ticket(g_);
  }
  /* the listed channels only (row i = ids[i]); every other channel of every member skips the call */
  uint64_t submit_host(const std::vector<uint32_t> &ids, const int16_t *I_or_X, const int16_t *Q, size_t in_pitch, void *audio, size_t out_pitch,
                       int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o = nullptr) {
    check(sdr_graph_submit_host(g_, ids.data(), (uint32_t)ids.size(), I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o),
          "sdr_graph_submit_host");
    return sdr_graph_host_ticket(g_);
  }
  void process_host(const int16_t *I_or_X, const int16_t *Q, size_t in_pitch, void *audio, size_t out_pitch, int out_fmt, uint32_t n_blocks,
                    const sdr_graph_outputs *o = nullptr) {
    check(sdr_graph_process_host(g_, nullptr, n_, I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o), "sdr_graph_process_host");
  }
  void process_host(const std::vector<uint32_t> &ids, const int16_t *I_or_X, const int16_t *Q, size_t in_pitch, void *audio, size_t out_pitch,
                    int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o = nullptr) {
    check(sdr_graph_process_host(g_, ids.data(), (uint32_t)ids.size(), I_or_X, Q, in_pitch, audio, out_pitch, out_fmt, n_blocks, o),
          "sdr_graph_process_host");
  }
  /* waterfall lines from the grabber tap (sdr_graph_attach_waterfall); the calls are then the _waterfall ones below */
  void attach_waterfall(WaterfallBatch *wf) { check(sdr_graph_attach_waterfall(g_, wf ? wf->handle() : nullptr), "sdr_graph_attach_waterfall"); }
  /* host lines [rows][wf.line_slots(n_blocks)][256] float, line_counts [rows] (may be null); ids empty: every channel */
  uint64_t submit_host(const std::vector<uint32_t> &ids, const int16_t *I_or_X, const int16_t *Q, size_t in_pitch, void *audio, size_t out_pitch,
                       int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o, float *lines, uint32_t *line_counts) {
    check(sdr_graph_submit_host_waterfall(g_, ids.empty() ? nullptr : ids.data(), ids.empty() ? n_ : (uint32_t)ids.size(), I_or_X, Q, in_pitch, audio,
                                          out_pitch, out_fmt, n_blocks, o, lines, line_counts),
          "sdr_graph_submit_host_waterfall");
    return sdr_graph_host_ticket(g_);
  }
  void process_host(const std::vector<uint32_t> &ids, const int16_t *I_or_X, const int16_t *Q, size_t in_pitch, void *audio, size_t out_pitch,
                    int out_fmt, uint32_t n_blocks, const sdr_graph_outputs *o, float *lines, uint32_t *line_counts) {
    check(sdr_graph_process_host_waterfall(g_, ids.empty() ? nullptr : ids.data(), ids.empty() ? n_ : (uint32_t)ids.size(), I_or_X, Q, in_pitch, audio,
                                           out_pitch, out_fmt, n_blocks, o, lines, line_counts),
          "sdr_graph_process_host_waterfall");
  }
  void wait_host() { check(sdr_graph_wait_host(g_), "sdr_graph_wait_host"); }
  void wait_host(uint64_t ticket) { check(sdr_graph_wait_host_ticket(g_, ticket), "sdr_graph_wait_host_ticket"); }
  sdr_graph_t *handle() { return g_; }

 private:
  static void check(int rc, const char *what) {
    if (rc != SDR_OK) throw std::runtime_error(std::string(what) + ": " + sdr_graph_last_error());
  }
  sdr_graph_t *g_;
  uint32_t n_;
};

}  // namespace sdr
#endif
