/* tests/cpp/grabber_snapshots_smoke.cpp -- the grabber's process overloads that return every published snapshot and its
 * spectrum (include/SdrAux.hpp, sdr_grabber_process_device_snapshots) compile against the C ABI and link to the product
 * library.  Without a GPU the constructor fails loudly (no CPU fallback); with one, 3 blocks of a constant run on all 4
 * channels, then 2 blocks on channels 3 and 1: the second call's slot 0 starts with the carried third block. */
#include <cstdio>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/SdrAux.hpp"

int main() {
  try {
    sdr::GrabberBatch gr(4);
    const size_t pitch = 3 * 128;
    std::vector<int16_t> h(2 * 4 * pitch);
    for (size_t i = 0; i < h.size(); i++) h[i] = (int16_t)(i % pitch < 256 ? 1 : 2); /* blocks 0, 1: 1; block 2: 2 */
    int16_t *d = nullptr, *snaps = nullptr;
    float *power = nullptr;
    if (cudaMalloc(&d, h.size() * sizeof(int16_t)) != cudaSuccess || cudaMalloc(&snaps, 4 * 2 * 512 * sizeof(int16_t)) != cudaSuccess ||
        cudaMalloc(&power, 4 * 2 * 256 * sizeof(float)) != cudaSuccess)
      throw std::runtime_error("cudaMalloc");
    cudaMemcpy(d, h.data(), h.size() * sizeof(int16_t), cudaMemcpyHostToDevice);
    uint32_t counts[4] = {9, 9, 9, 9};
    gr.process(d, d + 4 * pitch, pitch, 3, snaps, power, counts);
    const bool all_one = counts[0] == 1 && counts[3] == 1;
    gr.process({3, 1}, d, d + 4 * pitch, pitch, 2, nullptr, power, counts);
    std::vector<float> p(2 * 256);
    cudaMemcpy(p.data(), power, p.size() * sizeof(float), cudaMemcpyDeviceToHost);
    cudaDeviceSynchronize();
    cudaFree(d); cudaFree(snaps); cudaFree(power);
    /* slot 0 of the second call: the carried block of 2s, then a block of 1s: DC bin = (128 * 2 + 128 * 1)^2 * 2 */
    const bool ok = all_one && counts[0] == 1 && counts[1] == 1 && p[0] == 2.0f * 384.0f * 384.0f;
    std::printf("GPU_OK counts=%u,%u dc=%g\n", counts[0], counts[1], (double)p[0]);
    return ok ? 0 : 2;
  } catch (const std::runtime_error &e) {
    std::printf("NO_DEVICE %s\n", e.what());
    return 0;
  }
}
