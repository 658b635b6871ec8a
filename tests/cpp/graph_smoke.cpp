/* tests/cpp/graph_smoke.cpp -- the streamed receiver graph (include/SdrGraph.hpp, sdr_graph.h) compiles against the C ABI
 * and links to the product libraries.  Without a GPU the first constructor fails loudly (no CPU fallback); with one, 3 blocks
 * of a constant run through pre-processor -> grabber -> receiver on 4 channels from host memory: every row publishes one
 * snapshot, whose DC bin is that of a constant 7 + 7j, and a graph with mismatched channel counts is refused. */
#include <cstdio>
#include <vector>

#include "../../include/SdrGraph.hpp"

int main() {
  try {
    sdr::SdrBatch rx(4);
    sdr::PreProcessorBatch pp(4);
    sdr::GrabberBatch gr(4);
    sdr::SdrGraph graph(rx, &pp, nullptr, &gr);
    const uint32_t nb = 3;
    const size_t pitch = nb * 128;
    std::vector<int16_t> I(4 * pitch, 7), Q(4 * pitch, 7), audio(4 * pitch, 0);
    std::vector<float> power(4 * 2 * 256, -1.0f);
    uint32_t counts[4] = {9, 9, 9, 9};
    sdr_graph_outputs o = {nullptr, nullptr, power.data(), nullptr, counts};
    const uint64_t t = graph.submit_host(I.data(), Q.data(), pitch, audio.data(), pitch, SDR_FMT_I16, nb, &o);
    graph.wait_host(t);
    bool refused = false;
    {
      sdr::GrabberBatch other(5);
      try { sdr::SdrGraph bad(rx, nullptr, nullptr, &other); } catch (const std::runtime_error &) { refused = true; }
    }
    /* 256 samples of 7 + 7j: DC power = (256 * 7)^2 * 2; slot 1 of every row is past counts and keeps its -1 */
    const bool ok = t == 1 && counts[0] == 1 && counts[3] == 1 && power[0] == 2.0f * 1792.0f * 1792.0f && power[256] == -1.0f && refused;
    std::printf("GPU_OK ticket=%llu counts=%u dc=%g refused=%d\n", (unsigned long long)t, counts[0], (double)power[0], (int)refused);
    return ok ? 0 : 2;
  } catch (const std::runtime_error &e) {
    std::printf("NO_DEVICE %s\n", e.what());
    return 0;
  }
}
