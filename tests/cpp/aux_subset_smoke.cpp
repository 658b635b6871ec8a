/* tests/cpp/aux_subset_smoke.cpp -- the aux host classes' subset overloads and checkpoint calls compile against the C ABI and
 * link to the product library.  Without a GPU the constructor fails loudly (no CPU fallback); with one, channels 5 and 2
 * of the pre-processor and the I/Q generator run one block of silence while the others skip the call, and channel 5's
 * state moves to channel 0 of the grabber's neighbour handles. */
#include <cstdio>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/SdrAux.hpp"

int main() {
  try {
    sdr::PreProcessorBatch pp(8);
    sdr::IQGeneratorBatch iq(8);
    sdr::GrabberBatch gr(8);
    const std::vector<uint32_t> ids{5, 2};
    std::vector<int16_t> I(2 * 128, 0), Q(2 * 128, 0), oi(2 * 128, 1), oq(2 * 128, 1);
    pp.setI2SerrorCompensation(sdr::all, 1);
    pp.process_host(ids, I.data(), Q.data(), 128, oi.data(), oq.data(), 128, 1);
    iq.process_host(ids, I.data(), 128, oi.data(), oq.data(), 128, 1);
    int16_t *d = nullptr;
    if (cudaMalloc(&d, 2 * 2 * 128 * sizeof(int16_t)) != cudaSuccess) throw std::runtime_error("cudaMalloc");
    cudaMemset(d, 0, 2 * 2 * 128 * sizeof(int16_t));
    gr.process(ids, d, d + 2 * 128, 128, 1);
    cudaDeviceSynchronize();
    cudaFree(d);
    sdr::PreProcessorBatch pp2(3);
    sdr::IQGeneratorBatch iq2(3);
    sdr::GrabberBatch gr2(3);
    pp2.import_state({0}, pp.export_state({5}));
    iq2.import_state({0}, iq.export_state({5}));
    gr2.import_state({0}, gr.export_state({5}));
    const bool ok = oi[0] == 0 && oq[0] == 0 && pp2.getI2SerrorCompensation(0) == 1;
    std::printf("GPU_OK out0=%d corr=%d blob=%zu/%zu/%zu\n", (int)oi[0], (int)pp2.getI2SerrorCompensation(0), sdr::PreProcessorBatch::state_bytes(),
                sdr::IQGeneratorBatch::state_bytes(), sdr::GrabberBatch::state_bytes());
    return ok ? 0 : 2;
  } catch (const std::runtime_error &e) {
    std::printf("NO_DEVICE %s\n", e.what());
    return 0;
  }
}
