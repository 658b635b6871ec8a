/* tests/cpp/pp_block_status_smoke.cpp -- the pre-processor's records overloads (include/SdrAux.hpp, block_status) compile
 * against the C ABI and link to the product library.  Without a GPU the constructor fails loudly (no CPU fallback); with
 * one, every channel runs two blocks on host planes with records (channel 3 with correction +1), channel 3 alone one more
 * block, then channels 5 and 2 one block on device planes; the records are checked against the input and get_status. */
#include <cstdio>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/SdrAux.hpp"

int main() {
  try {
    sdr::PreProcessorBatch pp(8);
    pp.setI2SerrorCompensation(3u, 1);
    std::vector<int16_t> I(8 * 256), Q(8 * 256, 0), oi(8 * 256), oq(8 * 256);
    for (size_t k = 0; k < I.size(); k++) I[k] = (int16_t)(k % 1000);
    alignas(16) int32_t rec[2 * SDR_PP_BS_FIELDS * 8];
    pp.process_host(I.data(), Q.data(), 256, oi.data(), oq.data(), 256, 2, rec);
    alignas(16) int32_t rec1[SDR_PP_BS_FIELDS];
    pp.process_host(std::vector<uint32_t>{3}, I.data(), Q.data(), 128, oi.data(), oq.data(), 128, 1, rec1);
    int16_t *d = nullptr;
    int32_t *drec = nullptr;
    if (cudaMalloc(&d, 8 * 128 * sizeof(int16_t)) != cudaSuccess || cudaMalloc(&drec, 16 * sizeof(int32_t)) != cudaSuccess)
      throw std::runtime_error("cudaMalloc");
    cudaMemset(d, 0, 8 * 128 * sizeof(int16_t));
    pp.process({5, 2}, d, d + 2 * 128, 128, d + 4 * 128, d + 6 * 128, 128, 1, drec, nullptr);
    cudaDeviceSynchronize();
    cudaFree(d); cudaFree(drec);
    const sdr_preproc_status s = pp.status(3);
    const bool ok = rec[(1 * SDR_PP_BS_FIELDS + SDR_PP_BS_CORRECTION) * 8 + 3] == 1 &&
                    rec[(1 * SDR_PP_BS_FIELDS + SDR_PP_BS_SAVED_SAMPLE) * 8 + 3] == I[3 * 256 + 255] &&
                    rec1[SDR_PP_BS_SAVED_SAMPLE] == s.saved_sample && s.saved_sample == I[127];
    std::printf("GPU_OK saved=%d/%d\n", (int)rec1[SDR_PP_BS_SAVED_SAMPLE], (int)s.saved_sample);
    return ok ? 0 : 2;
  } catch (const std::runtime_error &e) {
    std::printf("NO_DEVICE %s\n", e.what());
    return 0;
  }
}
