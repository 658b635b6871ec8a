/* tests/cpp/subset_class_smoke.cpp -- the C++ host class's subset overloads compile against the C ABI and link to the product
 * library.  Without a GPU the constructor fails loudly (no CPU fallback); with one, channel 5 alone runs one block of silence
 * while the other channels skip the call. */
#include <cstdio>
#include <vector>
#include "../../include/SdrBatch.hpp"

int main() {
  try {
    sdr::SdrBatch sdr(8);
    std::vector<int16_t> I(2 * 128, 0), Q(2 * 128, 0), out(2 * 128, 1);
    std::vector<uint32_t> rec((size_t)SDR_BS_FIELDS * 2 + 4);
    uint32_t *r = rec.data() + ((16 - ((uintptr_t)rec.data() & 15)) & 15) / 4; /* 16-byte aligned */
    const std::vector<uint32_t> ids{5, 2};
    sdr.process_host(ids, I.data(), Q.data(), 128, SDR_FMT_I16, out.data(), 128, SDR_FMT_I16, 1, r);
    sdr.submit_host(std::vector<uint32_t>{7}, I.data(), Q.data(), 128, SDR_FMT_I16, out.data(), 128, SDR_FMT_I16, 1);
    sdr.wait_host();
    std::printf("GPU_OK out0=%d gain=%g\n", (int)out[0], (double)reinterpret_cast<const float *>(r)[0]);
    return out[0] == 0 ? 0 : 2;
  } catch (const std::runtime_error &e) {
    std::printf("NO_DEVICE %s\n", e.what());
    return 0;
  }
}
