/* tests/cpp/waterfall_smoke.cpp -- the waterfall wrappers (include/SdrAux.hpp WaterfallBatch and the grabber overload,
 * include/SdrGraph.hpp attach_waterfall and the _waterfall calls) compile against the C ABI and link to the product
 * libraries.  Without a GPU the first constructor fails loudly (no CPU fallback); with one, K = 2 over 2 channels: a call of 3
 * blocks completes one pair per channel (no line yet), a call of 2 more blocks completes the second pair: one line, whose DC
 * bin is the mean of the two pairs' DC power. */
#include <cstdio>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/SdrGraph.hpp"

int main() {
  try {
    sdr::GrabberBatch gr(2);
    sdr::WaterfallBatch wf(2, 2);
    const size_t pitch = 3 * 128;
    std::vector<int16_t> h(2 * 2 * pitch, 1); /* every sample 1 */
    int16_t *d = nullptr;
    float *lines = nullptr;
    if (cudaMalloc(&d, h.size() * sizeof(int16_t)) != cudaSuccess || cudaMalloc(&lines, 2 * 1 * 256 * sizeof(float)) != cudaSuccess)
      throw std::runtime_error("cudaMalloc");
    cudaMemcpy(d, h.data(), h.size() * sizeof(int16_t), cudaMemcpyHostToDevice);
    uint32_t counts[2] = {9, 9};
    gr.process(wf, {}, d, d + 2 * pitch, pitch, 3, lines, counts); /* Lmax = (1 + 2) / 2 = 1 */
    const bool none = counts[0] == 0 && counts[1] == 0;
    gr.process(wf, {1, 0}, d, d + 2 * pitch, pitch, 2, lines, counts);
    std::vector<float> p(2 * 256);
    cudaMemcpy(p.data(), lines, p.size() * sizeof(float), cudaMemcpyDeviceToHost);
    const std::vector<uint8_t> blob = wf.export_state({0});
    cudaFree(d); cudaFree(lines);
    /* both pairs: 256 points of (1, 1): DC power = 256^2 * 2 */
    const bool ok = none && counts[0] == 1 && counts[1] == 1 && p[0] == 2.0f * 256.0f * 256.0f && blob.size() == sdr::WaterfallBatch::state_bytes();
    std::printf("GPU_OK counts=%u,%u dc=%g lmax=%u\n", counts[0], counts[1], (double)p[0], wf.line_slots(2));
    return ok ? 0 : 2;
  } catch (const std::runtime_error &e) {
    std::printf("NO_DEVICE %s\n", e.what());
    return 0;
  }
}
