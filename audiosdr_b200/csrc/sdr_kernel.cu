/* sdr_kernel.cu -- launch dispatch and the small kernels around the receiver pipeline (state reset / fill / gather,
 * FP32 roofline microbenchmark, self-tests).
 *
 * The pipeline kernel itself -- one CTA per 32-channel group, one warp per pipeline stage of the launch's bucket
 * (sdr_pipeline.cuh, sdr_lay.h) -- is compiled once per tile length in sdr_pipe_t32.cu / _t16.cu / _t8.cu.  Build flags matter
 * for parity: -fmad=false (no FMA contraction; the reference rounds every product and sum separately), IEEE division
 * and square root (nvcc defaults), no FTZ.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "sdr_kernel.h"
#include "sdr_pipeline.cuh"

using namespace sdrk;

extern "C" {
int sdrk_setup_pipe_t32(const float *), sdrk_setup_pipe_t16(const float *), sdrk_setup_pipe_t8(const float *), sdrk_setup_pipe_t32c(const float *);
int sdrk_launch_pipe_t32(const SdrLaunch *, void *), sdrk_launch_pipe_t16(const SdrLaunch *, void *), sdrk_launch_pipe_t8(const SdrLaunch *, void *);
int sdrk_launch_pipe_t32c(const SdrLaunch *, void *);
int sdrk_setup_pipe_t32s(const float *), sdrk_launch_pipe_t32s(const SdrLaunch *, void *), sdrk_occupancy_t32s(const SdrLaunch *);
int sdrk_occupancy_t32(const SdrLaunch *), sdrk_occupancy_t16(const SdrLaunch *), sdrk_occupancy_t8(const SdrLaunch *);
int sdrk_setup_als_pass(void), sdrk_occupancy_als_pass(const SdrLaunch *); /* sdr_als_pass.cu */
}

/* Zero (or re-seed) state words of listed channels: the side effects of the reference setters that
 * re-initialise filter state / rings (SURVEY 8a13), and the turn of a lagging channel's blanker slots.  One thread per
 * (entry, word). */
extern "C" __global__ void sdr_reset_kernel(float *state, unsigned long long ch_stride, const uint32_t *chan, const uint32_t *mask,
                                            uint32_t n) {
  const uint32_t e = blockIdx.y;
  if (e >= n) return;
  const uint32_t c = chan[e], m = mask[e];
  for (uint32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < SDR_STATE_WORDS; w += gridDim.x * blockDim.x) {
    bool z = false;
    if ((m & SDRK_R_IF) && w >= W_IF_I && w < W_IF_Q + 16) z = true;
    if ((m & SDRK_R_IMG) && w >= W_IMG_I && w < W_IMG_Q + 16) z = true;
    if ((m & SDRK_R_AUD) && w >= W_AUD && w < W_AUD + 16) z = true;
    if ((m & SDRK_R_ALS) && w >= W_ALS_C && w < W_ALS_H + 128) z = true;
    if ((m & SDRK_R_NB) && w >= W_NB_MASK && w < W_NB_RING) z = true;
    if (z) state[(size_t)w * ch_stride + c] = 0.0f;
  }
  if (m & SDRK_R_NB) { /* the ring planes are float4 groups: group f of channel c is float4 number f*ch_stride + c */
    float4 *ring = reinterpret_cast<float4 *>(state + (size_t)W_NB_RING * ch_stride);
    for (uint32_t f = blockIdx.x * blockDim.x + threadIdx.x; f < 288; f += gridDim.x * blockDim.x)
      ring[(size_t)f * ch_stride + c] = make_float4(0.f, 0.f, 0.f, 0.f);
  } else if (m & (SDRK_R_TURN1 | SDRK_R_TURN2)) {
    /* task j < 32: mask word j of the 3 slots; task 32 + 32 * plane + g: float4 group g of the 3 slots of a ring plane */
    const uint32_t d = (m & SDRK_R_TURN1) ? 1u : 2u;
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < 128; j += gridDim.x * blockDim.x) {
      if (j < 32) {
        float v[3];
        for (uint32_t s = 0; s < 3; s++) v[s] = state[(size_t)(W_NB_MASK + s * 32 + j) * ch_stride + c];
        for (uint32_t s = 0; s < 3; s++) state[(size_t)(W_NB_MASK + (s + d) % 3 * 32 + j) * ch_stride + c] = v[s];
      } else {
        float4 *ring = reinterpret_cast<float4 *>(state + (size_t)W_NB_RING * ch_stride);
        const uint32_t pl = (j - 32) >> 5, g = j & 31;
        float4 v[3];
        for (uint32_t s = 0; s < 3; s++) v[s] = ring[(size_t)(pl * 96 + s * 32 + g) * ch_stride + c];
        for (uint32_t s = 0; s < 3; s++) ring[(size_t)(pl * 96 + (s + d) % 3 * 32 + g) * ch_stride + c] = v[s];
      }
    }
  }
}

/* state word `w` of every channel := v (used once at create for non-zero power-on values) */
extern "C" __global__ void sdr_fill_word_kernel(float *state, unsigned long long ch_stride, uint32_t w, float v, uint32_t n_ch) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < n_ch) state[(size_t)w * ch_stride + c] = v;
}

/* Address of state word `w` of channel `c`.  Words below W_NB_RING are stored channel-fastest; the blanker ring words
 * (plane, block slot, sample) are stored as float4 groups (sdr_pipeline.cuh, nb_group): word W_NB_RING + r is component r % 4 of
 * group r / 4. */
__device__ __forceinline__ size_t state_index(uint32_t w, uint32_t c, unsigned long long ch_stride) {
  if (w < W_NB_RING) return (size_t)w * ch_stride + c;
  const uint32_t r = w - W_NB_RING;
  return (size_t)W_NB_RING * ch_stride + ((size_t)(r >> 2) * ch_stride + c) * 4 + (r & 3u);
}

/* gather `n_words` listed state words (all SDR_STATE_WORDS in order if `words` is null) of `n` listed channels into out[n][n_words] */
extern "C" __global__ void sdr_gather_kernel(const float *state, unsigned long long ch_stride, const uint32_t *chan, uint32_t n,
                                             const uint32_t *words, uint32_t n_words, float *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)n * n_words) return;
  const uint32_t e = (uint32_t)(i / n_words), k = (uint32_t)(i % n_words);
  const uint32_t c = chan ? chan[e] : e;
  out[i] = state[state_index(words ? words[k] : k, c, ch_stride)];
}

/* the reverse: in[n][SDR_STATE_WORDS] -> the state words of `n` listed channels (checkpoint import) */
extern "C" __global__ void sdr_scatter_kernel(float *state, unsigned long long ch_stride, const uint32_t *chan, uint32_t n, const float *in) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)n * SDR_STATE_WORDS) return;
  const uint32_t e = (uint32_t)(i / SDR_STATE_WORDS), k = (uint32_t)(i % SDR_STATE_WORDS);
  state[state_index(k, chan[e], ch_stride)] = in[i];
}

extern "C" int sdrk_setup_device(const float *hilbert64) {
  int e = sdrk_setup_pipe_t32(hilbert64);
  if (!e) e = sdrk_setup_pipe_t16(hilbert64);
  if (!e) e = sdrk_setup_pipe_t8(hilbert64);
  if (!e) e = sdrk_setup_pipe_t32c(hilbert64);
  if (!e) e = sdrk_setup_pipe_t32s(hilbert64);
  if (!e) e = sdrk_setup_als_pass();
  return e;
}

extern "C" int sdrk_launch_pipeline(const SdrLaunch *L, void *stream) {
  if (L->n_groups == 0) return 0;
  if (L->lay.T == 32) {
    if (L->flags & SDRL_CONTRACT) return sdrk_launch_pipe_t32c(L, stream);
    static const bool general = [] { const char *e = getenv("SDR_NO_CLASS_KERNEL"); return e && e[0] == '1'; }(); /* A/B switch */
    return L->lay.cls == CLS_SSB && !general ? sdrk_launch_pipe_t32s(L, stream) : sdrk_launch_pipe_t32(L, stream);
  }
  if (L->lay.T == 16) return sdrk_launch_pipe_t16(L, stream);
  if (L->lay.T == 8) return sdrk_launch_pipe_t8(L, stream);
  return 1;
}

extern "C" int sdrk_occupancy(const SdrLaunch *L) {
  if (L->lay.cls == CLS_ALS) return sdrk_occupancy_als_pass(L);
  return L->lay.T == 32 ? (L->lay.cls == CLS_SSB ? sdrk_occupancy_t32s(L) : sdrk_occupancy_t32(L)) : (L->lay.T == 16 ? sdrk_occupancy_t16(L) : sdrk_occupancy_t8(L));
}

extern "C" int sdrk_launch_reset(float *state, unsigned long long ch_stride, const uint32_t *chan, const uint32_t *mask, uint32_t n,
                                 void *stream) {
  if (n == 0) return 0;
  dim3 grid(4, n);
  sdr_reset_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(state, ch_stride, chan, mask, n);
  return (int)cudaGetLastError();
}

extern "C" int sdrk_launch_fill_word(float *state, unsigned long long ch_stride, uint32_t w, float v, uint32_t n_ch, void *stream) {
  sdr_fill_word_kernel<<<(n_ch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(state, ch_stride, w, v, n_ch);
  return (int)cudaGetLastError();
}

extern "C" int sdrk_launch_gather(const float *state, unsigned long long ch_stride, const uint32_t *chan, uint32_t n,
                                  const uint32_t *words, uint32_t n_words, float *out, void *stream) {
  const size_t tot = (size_t)n * n_words;
  if (tot == 0) return 0;
  sdr_gather_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(state, ch_stride, chan, n, words, n_words, out);
  return (int)cudaGetLastError();
}

extern "C" int sdrk_launch_scatter(float *state, unsigned long long ch_stride, const uint32_t *chan, uint32_t n, const float *in, void *stream) {
  const size_t tot = (size_t)n * SDR_STATE_WORDS;
  if (tot == 0) return 0;
  sdr_scatter_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, (cudaStream_t)stream>>>(state, ch_stride, chan, n, in);
  return (int)cudaGetLastError();
}

/* ---- FP32 pipe microbenchmark: the denominator of the FP32 roofline (MEASURED_PEAKS.json has no FP32 entry).
 * kind 0: dependent FFMA chains (2 flop / instruction, what a contracting build could reach);
 * kind 1: alternating FMUL / FADD chains (1 flop / instruction: the instruction mix this parity-exact build issues).
 * 8 independent chains per thread hide the 4-cycle pipe latency. */
template <int KIND>
__global__ void __launch_bounds__(256) sdr_fp32_peak_kernel(float *out, int iters, float a, float b) {
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = a + (float)(threadIdx.x + i);
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int u = 0; u < 8; u++) {
#pragma unroll
      for (int i = 0; i < 8; i++) {
        if (KIND == 0) v[i] = __fmaf_rn(v[i], a, b);
        else if (KIND == 1) { v[i] = __fmul_rn(v[i], a); v[i] = __fadd_rn(v[i], b); }
        else v[i] = (float)__fma_rn((double)v[i], (double)a, (double)b); /* KIND 2: F2F + DFMA + F2F per element */
      }
    }
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; i++) s += v[i];
  if (s == 123.456f) out[0] = s; /* keep the chains alive */
}

/* returns instructions/s (FP32-pipe lane-instructions per second) in *lane_ips and elapsed ms; 0 on success */
extern "C" int sdrk_fp32_peak(int kind, int iters, double *lane_ips, float *ms_out) {
  float *d = nullptr;
  if (cudaMalloc(&d, 4) != cudaSuccess) return 1;
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int grid = sms * 8, block = 256;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 2; rep++) { /* first pass warms up */
    cudaEventRecord(e0);
    if (kind == 0) sdr_fp32_peak_kernel<0><<<grid, block>>>(d, iters, 0.999f, 0.001f);
    else if (kind == 1) sdr_fp32_peak_kernel<1><<<grid, block>>>(d, iters, 0.999f, 0.001f);
    else sdr_fp32_peak_kernel<2><<<grid, block>>>(d, iters, 0.999f, 0.001f);
    cudaEventRecord(e1);
    if (cudaEventSynchronize(e1) != cudaSuccess) { cudaFree(d); return 2; }
  }
  float ms = 0.f;
  cudaEventElapsedTime(&ms, e0, e1);
  const double instr = (double)grid * block * (double)iters * 64.0 * (kind == 1 ? 2.0 : 1.0); /* kind 2 counts DFMAs */
  *lane_ips = instr / (ms * 1e-3);
  *ms_out = ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(d);
  return 0;
}

/* ---- self-test: the batched branch-free envelope (sqrt_hack_batch) against the plain IEEE-divide form (sqrt_hack),
 * bit for bit, over `n` float bit patterns starting at `first` with stride `step` (covers every exponent). */
__global__ void sdr_selftest_envelope_kernel(unsigned first, unsigned step, unsigned long long n, unsigned long long *bad) {
  unsigned long long i = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 8ull;
  unsigned long long local = 0;
  for (; i < n; i += (unsigned long long)gridDim.x * blockDim.x * 8ull) {
    float x[8], e[8];
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = fabsf(__uint_as_float(first + (unsigned)((i + k) * step)));
    sqrt_hack_batch<8>(x, e);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const float w = sqrt_hack(x[k]);
      const bool same = __float_as_uint(w) == __float_as_uint(e[k]) || (w != w && e[k] != e[k]);
      if (!same) local++;
    }
  }
  if (local) atomicAdd(bad, local);
}

/* ---- self-test: div_inrange (the PLL's division without range check and slow-path branch) against the IEEE divide, bit for
 * bit, over `n` pseudo-random operand pairs of both signs whose magnitudes cover [2^-60, 2^60] exponent by exponent
 * (mantissas from a 64-bit mix of the pair index; every 16th pair sits on a power of two or one ulp beside it). */
__global__ void sdr_selftest_divide_kernel(unsigned long long seed, unsigned long long n, unsigned long long *bad) {
  unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long local = 0;
  for (; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    unsigned long long z = seed + i * 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; z ^= z >> 31;
    unsigned ma = (unsigned)z & 0x7FFFFFu, mb = (unsigned)(z >> 23) & 0x7FFFFFu;
    const unsigned ea = 67u + (unsigned)((z >> 46) % 121u), eb = 67u + (unsigned)((z >> 54) % 121u); /* 2^-60 .. 2^60 */
    if ((i & 15ull) == 0) { ma = (z >> 62) & 1 ? 0u : 0x7FFFFFu; mb = (z >> 63) ? 0u : 1u; }
    if (ea == 187u) ma = 0; /* 2^60 itself is the upper end */
    if (eb == 187u) mb = 0;
    const float a = __uint_as_float(((unsigned)(i & 1) << 31) | (ea << 23) | ma);
    const float b = __uint_as_float(((unsigned)((i >> 1) & 1) << 31) | (eb << 23) | mb);
    if (__float_as_uint(div_inrange(a, b)) != __float_as_uint(__fdiv_rn(a, b))) local++;
  }
  if (local) atomicAdd(bad, local);
}

extern "C" int sdrk_selftest_divide(unsigned long long seed, unsigned long long n, unsigned long long *mismatches) {
  unsigned long long *d = nullptr;
  if (cudaMalloc(&d, 8) != cudaSuccess) return 1;
  cudaMemset(d, 0, 8);
  sdr_selftest_divide_kernel<<<148 * 8, 256>>>(seed, n, d);
  cudaError_t e = cudaMemcpy(mismatches, d, 8, cudaMemcpyDeviceToHost);
  cudaFree(d);
  return e == cudaSuccess ? 0 : 2;
}

extern "C" int sdrk_selftest_envelope(unsigned first, unsigned step, unsigned long long n, unsigned long long *mismatches) {
  unsigned long long *d = nullptr;
  if (cudaMalloc(&d, 8) != cudaSuccess) return 1;
  cudaMemset(d, 0, 8);
  sdr_selftest_envelope_kernel<<<148 * 8, 256>>>(first, step, n, d);
  cudaError_t e = cudaMemcpy(mismatches, d, 8, cudaMemcpyDeviceToHost);
  cudaFree(d);
  return e == cudaSuccess ? 0 : 2;
}
