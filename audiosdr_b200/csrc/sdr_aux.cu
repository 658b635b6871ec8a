/* sdr_aux.cu -- the two blocks either side of the receiver chain, batched (SURVEY.md 8f rows 2 and 4): kernels and the C ABI
 * of include/sdr_aux.h.  Per-lane arithmetic lives in sdr_aux_core.cuh (also run on the host by tests/emu/aux_emu.cpp).
 *
 *  I/Q generator (AudioIQgenerator.cpp:33-87): a 257-tap Hilbert FIR in its 64-product compact form plus a 128-sample delay,
 *    purely feed-forward, so the kernel is parallel over channels AND time: one CTA = one channel x 4096 outputs, the
 *    input span (+256 history) converted to float once into shared memory, one lane = 16 consecutive outputs with two
 *    sliding 16-register windows.  192 unfused FP32 operations per output sample against 6 bytes of traffic: FP32-issue
 *    bound.  History (the last 256 inputs per channel) is the only state, kept in two alternating buffers.
 *  Pre-processor (AudioSDRpreProcessor.cpp:46-138): with the detector off a channel is a one-sample shift and/or a swap --
 *    a feed-forward copy, 8 bytes moved per sample, HBM bound (pp_static_kernel).  Channels whose detector is running are
 *    compacted into a list and handled block by block by pp_detect_kernel (lane = channel, 128-point FFT per block in
 *    shared memory), because their correction may change from one block to the next.
 *  Both blocks serve calls on every channel and on subsets (compact planes, row r = channel ids[r]) with one kernel template
 *  per job; the two forms differ only in where a row's channel comes from (see kList below).
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/sdr_aux.h"
#include "aux_tables.inc"
#include "sdr_aux_core.cuh"

__constant__ float c_iq_h[64];
__constant__ float c_fft_tw[128];
__constant__ float c_fft_tw256[256];

/* The pre-processor and I/Q generator kernels are templates on kList, one source per job.  kList = true serves the *_subset
 * entry points: the planes are compact, row r belonging to channel ids[r] (device copy of the call's id list), and
 * L.n_channels counts rows.  Plane addresses use r; state (history, gains, PpState) uses ch = kList ? ids[r] : r.
 * kList = false is the call on every channel (row = channel, ids unused). */

/* ================================================================== I/Q generator ==== */
#define IQ_SEG 4096
#define IQ_THREADS 256
#define IQ_XS_WORDS (IQ_SEG + 256 + (IQ_SEG + 256) / 16 + 16)

struct IqLaunch {
  const int16_t *x; int16_t *oi, *oq;
  unsigned long long in_pitch, out_pitch;
  const int16_t *hist_in; int16_t *hist_out; /* [n_channels][256] */
  const float2 *gains;                       /* (gainI, gainQ) per channel */
  uint32_t n_samples, n_channels, segs;
};

__device__ __forceinline__ void iq_unpack8(const int4 v, float *f) {
  const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; i++) {
    f[2 * i] = aux_q15_to_float((int)(int16_t)(w[i] & 0xFFFF));
    f[2 * i + 1] = aux_q15_to_float(w[i] >> 16);
  }
}

template <bool kList>
__global__ void __launch_bounds__(IQ_THREADS) iq_generate_kernel(const IqLaunch L, const uint32_t *ids) {
  __shared__ float xs[IQ_XS_WORDS];
  const uint32_t r = blockIdx.x / L.segs, seg = blockIdx.x % L.segs, ch = kList ? __ldg(ids + r) : r;
  const long base = (long)seg * IQ_SEG;
  const int16_t *row = L.x + (size_t)r * L.in_pitch;
  /* the span [base-256, base+SEG) as floats at padded positions; 8 samples (16 bytes) per thread and pass */
  for (int t = threadIdx.x; t < (IQ_SEG + 256) / 8; t += IQ_THREADS) {
    const long n = base - 256 + 8 * t;
    int4 v = make_int4(0, 0, 0, 0);
    if (n < 0) v = *reinterpret_cast<const int4 *>(L.hist_in + (size_t)ch * 256 + (256 + n));
    else if (n < (long)L.n_samples) v = __ldg(reinterpret_cast<const int4 *>(row + n));
    float f[8];
    iq_unpack8(v, f);
    float *dst = xs + 8 * t + ((8 * t) >> 4);
#pragma unroll
    for (int i = 0; i < 8; i++) dst[i] = f[i];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long n0 = base + 512 * warp + 16 * lane;
  if (n0 >= (long)L.n_samples) return;
  const int q0 = 256 + 512 * warp + 16 * lane;
  float acc[16];
  iq_lane_fir(xs, q0, c_iq_h, acc);
  const float2 g = L.gains[ch];
  uint32_t wi[8], wq[8];
  if (g.x == 1.0f && g.y == 1.0f) { /* the constructor's balance (IQ.h:72-73): uniform over the CTA, no FP64, no range test */
#pragma unroll
    for (int c = 0; c < 16; c += 2) {
      const int i0 = aux_to_pcm_unit(iq_lane_delayed(xs, q0, c)), i1 = aux_to_pcm_unit(iq_lane_delayed(xs, q0, c + 1));
      const int q0v = aux_to_pcm_unit(acc[c]), q1v = aux_to_pcm_unit(acc[c + 1]);
      wi[c >> 1] = ((uint32_t)i0 & 0xFFFFu) | ((uint32_t)i1 << 16);
      wq[c >> 1] = ((uint32_t)q0v & 0xFFFFu) | ((uint32_t)q1v << 16);
    }
  } else {
#pragma unroll
    for (int c = 0; c < 16; c += 2) {
      const int i0 = aux_to_pcm(iq_lane_delayed(xs, q0, c), g.x), i1 = aux_to_pcm(iq_lane_delayed(xs, q0, c + 1), g.x);
      const int q0v = aux_to_pcm(acc[c], g.y), q1v = aux_to_pcm(acc[c + 1], g.y);
      wi[c >> 1] = ((uint32_t)i0 & 0xFFFFu) | ((uint32_t)i1 << 16);
      wq[c >> 1] = ((uint32_t)q0v & 0xFFFFu) | ((uint32_t)q1v << 16);
    }
  }
  uint4 *di = reinterpret_cast<uint4 *>(L.oi + (size_t)r * L.out_pitch + n0);
  uint4 *dq = reinterpret_cast<uint4 *>(L.oq + (size_t)r * L.out_pitch + n0);
  di[0] = make_uint4(wi[0], wi[1], wi[2], wi[3]); di[1] = make_uint4(wi[4], wi[5], wi[6], wi[7]);
  dq[0] = make_uint4(wq[0], wq[1], wq[2], wq[3]); dq[1] = make_uint4(wq[4], wq[5], wq[6], wq[7]);
}

/* the last 256 inputs of every listed channel become the next call's history.  Calls on every channel write the other
 * buffer (no ordering hazard).  Subset calls rewrite it IN PLACE (hist_out == hist_in), because the channels that skip the
 * call keep theirs in the same buffer: one warp = one row, and with fewer than 256 new samples lane j reads the old slot
 * that lane j + n_samples/8 overwrites, so every lane loads before any lane stores. */
template <bool kList>
__global__ void iq_history_kernel(const IqLaunch L, const uint32_t *ids) {
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t r = idx >> 5, j = idx & 31;
  if (r >= L.n_channels) return; /* whole warps */
  const uint32_t ch = kList ? __ldg(ids + r) : r;
  const long n = (long)L.n_samples - 256 + 8 * (long)j;
  int4 v;
  if (n < 0) v = *reinterpret_cast<const int4 *>(L.hist_in + (size_t)ch * 256 + (256 + n));
  else v = __ldg(reinterpret_cast<const int4 *>(L.x + (size_t)r * L.in_pitch + n));
  if (kList) __syncwarp();
  *reinterpret_cast<int4 *>(L.hist_out + (size_t)ch * 256 + 8 * j) = v;
}

/* ================================================================== pre-processor ==== */
struct PpLaunch {
  const int16_t *I, *Q; int16_t *oi, *oq;
  unsigned long long in_pitch, out_pitch;
  PpState *state;
  uint32_t n_channels, n_blocks;
  uint32_t *auto_list, *auto_count;
};

__global__ void pp_apply_kernel(PpState *st, uint32_t n_channels, const PpSetterCall *calls, uint32_t n_calls) {
  const uint32_t ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= n_channels) return;
  PpState s = st[ch];
  for (uint32_t k = 0; k < n_calls; k++) {
    const PpSetterCall c = calls[k];
    if (c.channel == ch || c.channel == 0xFFFFFFFFu) pp_apply(s, c.setter, c.arg);
  }
  st[ch] = s;
}

/* the rows whose detector is running */
template <bool kList>
__global__ void pp_list_kernel(const PpLaunch L, const uint32_t *ids) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= L.n_channels) return;
  if (L.state[kList ? __ldg(ids + r) : r].autod) L.auto_list[atomicAdd(L.auto_count, 1u)] = r;
}

__device__ __forceinline__ void unpack_i16x8(const int4 v, int16_t *o) {
  const int w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int i = 0; i < 4; i++) { o[2 * i] = (int16_t)(w[i] & 0xFFFF); o[2 * i + 1] = (int16_t)(w[i] >> 16); }
}
__device__ __forceinline__ int4 pack_i16x8(const int16_t *o) {
  int w[4];
#pragma unroll
  for (int i = 0; i < 4; i++) w[i] = (int)(((uint32_t)(uint16_t)o[2 * i]) | ((uint32_t)(uint16_t)o[2 * i + 1] << 16));
  return make_int4(w[0], w[1], w[2], w[3]);
}

/* detector off: one thread = one 16-byte chunk of both rails.  8 bytes in + 8 bytes out per 2 samples... i.e. 8 B/sample. */
template <bool kList>
__global__ void __launch_bounds__(256) pp_static_kernel(const PpLaunch L, const uint32_t *ids) {
  const uint32_t chunks = L.n_blocks * 16; /* per channel */
  const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t r = (uint32_t)(idx / chunks), j = (uint32_t)(idx % chunks);
  if (r >= L.n_channels) return;
  const PpState s = L.state[kList ? __ldg(ids + r) : r];
  if (s.autod) return; /* pp_detect_kernel owns this channel for the call */
  const int16_t *ri = L.I + (size_t)r * L.in_pitch, *rq = L.Q + (size_t)r * L.in_pitch;
  const size_t n = (size_t)j * 8;
  const int4 a = __ldg(reinterpret_cast<const int4 *>(ri + n)), b = __ldg(reinterpret_cast<const int4 *>(rq + n));
  int4 oa = a, ob = b;
  if (s.corr != 0) {
    int16_t vi[8], vq[8], oi[8], oq[8];
    unpack_i16x8(a, vi); unpack_i16x8(b, vq);
    int16_t pi = (int16_t)s.saved, pq = (int16_t)s.saved;
    if (j) { if (s.corr == 1) pi = ri[n - 1]; else pq = rq[n - 1]; }
    pp_static_chunk(vi, vq, pi, pq, (j & 15) == 0, s.corr, 0, oi, oq);
    oa = pack_i16x8(oi); ob = pack_i16x8(oq);
  }
  int4 *di = reinterpret_cast<int4 *>(L.oi + (size_t)r * L.out_pitch + n), *dq = reinterpret_cast<int4 *>(L.oq + (size_t)r * L.out_pitch + n);
  *di = s.swap ? ob : oa;
  *dq = s.swap ? oa : ob;
}

/* detector off: savedSample after the call = the delayed rail's last input sample (PP.cpp:62-65 / 67-70).
 * kRec: the per-block records of these rows instead (sdr_preproc_process_device_status), one thread per (block, row), rows
 * fastest, so that each word's stores are coalesced across rows and the blocks of a row run in parallel (one thread per row
 * looping over the blocks measured 2.1x the plain call's time on the feed-forward path, DESIGN section 10).  Only the saved
 * sample moves: after block b it is the delayed rail's sample 128 b + 127, unchanged when the correction is 0; the thread of
 * the last block stores it in the state.  Rows with the detector on belong to pp_detect_kernel, which runs after this kernel
 * and changes their state. */
template <bool kList, bool kRec>
__global__ void pp_finish_kernel(const PpLaunch L, const uint32_t *ids, int32_t *rec) {
  if (kRec) {
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t n = L.n_channels, r = (uint32_t)(idx % n), b = (uint32_t)(idx / n);
    if (b >= L.n_blocks) return;
    const uint32_t ch = kList ? __ldg(ids + r) : r;
    const PpState s = L.state[ch]; /* the saved sample read here is used only when the correction is 0: never written then */
    if (s.autod) return;
    const size_t at = (size_t)r * L.in_pitch + (size_t)b * 128 + 127;
    const int32_t saved = s.corr == 1 ? (int32_t)L.I[at] : s.corr == -1 ? (int32_t)L.Q[at] : s.saved;
    int32_t *o = rec + (size_t)b * SDR_PP_BS_FIELDS * n + r;
    o[SDR_PP_BS_AUTO_DETECT * (size_t)n] = 0; o[SDR_PP_BS_CORRECTION * (size_t)n] = s.corr;
    o[SDR_PP_BS_FAILURE_COUNT * (size_t)n] = s.fail; o[SDR_PP_BS_SUCCESS_COUNT * (size_t)n] = s.succ;
    o[SDR_PP_BS_SAVED_SAMPLE * (size_t)n] = saved; o[SDR_PP_BS_SWAP * (size_t)n] = s.swap;
    if (b == L.n_blocks - 1 && s.corr != 0) L.state[ch].saved = saved;
    return;
  }
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= L.n_channels) return;
  const uint32_t ch = kList ? __ldg(ids + r) : r;
  const PpState s = L.state[ch];
  if (s.autod || s.corr == 0) return;
  const size_t last = (size_t)L.n_blocks * 128 - 1;
  L.state[ch].saved = (s.corr == 1 ? L.I : L.Q)[(size_t)r * L.in_pitch + last];
}

/* detector running: one CTA = 32 listed rows (lane = row) x PP_W warps that share each channel's work, block
 * after block.  Rows are staged through shared memory with whole-row (coalesced) transfers; a lane's row is 65 words from
 * its neighbour's (odd: no bank conflicts); the FFT buffer is [256][32] floats, lane-interleaved.  Warp 0 owns the
 * per-channel state (correction, counters); the butterflies of a stage, the conversions and the rows are split over
 * the warps with a CTA barrier between dependent phases.  kRec: warp 0 also stores each lane's state after every block
 * (sdr_preproc_process_device_status), column = the lane's plane row; padding lanes store nothing. */
#define PP_W 8
#define PP_ROW_WORDS 65
#define PP_DETECT_SMEM (256 * 32 * 4 + 2 * 32 * PP_ROW_WORDS * 4 + 2 * 32 * 4)
template <bool kList, bool kRec>
__global__ void __launch_bounds__(32 * PP_W) pp_detect_kernel(const PpLaunch L, const uint32_t *ids, int32_t *rec) {
  extern __shared__ __align__(16) unsigned char sm[];
  float *fft = reinterpret_cast<float *>(sm);
  uint32_t *rowI = reinterpret_cast<uint32_t *>(sm + 256 * 32 * 4), *rowQ = rowI + 32 * PP_ROW_WORDS;
  int *sh_det = reinterpret_cast<int *>(rowQ + 32 * PP_ROW_WORDS), *sh_swap = sh_det + 32;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const uint32_t n_auto = *L.auto_count, first = blockIdx.x * 32;
  if (first >= n_auto) return;
  const int row = first + lane < n_auto ? (int)L.auto_list[first + lane] : -1; /* the list holds plane rows */
  const int ch = kList && row >= 0 ? (int)__ldg(ids + row) : row;
  PpState s;
  s.corr = s.saved = s.fail = s.succ = s.swap = s.autod = s.pad0 = s.pad1 = 0;
  if (ch >= 0) s = L.state[ch]; /* every warp reads it; only warp 0's copy evolves and is written back */
  float *mine = fft + lane;
  for (uint32_t b = 0; b < L.n_blocks; b++) {
    for (int r = w; r < 32; r += PP_W) {
      const int rr = __shfl_sync(0xFFFFFFFFu, row, r);
      if (rr >= 0) {
        const uint32_t *si = reinterpret_cast<const uint32_t *>(L.I + (size_t)rr * L.in_pitch + (size_t)b * 128);
        const uint32_t *sq = reinterpret_cast<const uint32_t *>(L.Q + (size_t)rr * L.in_pitch + (size_t)b * 128);
        rowI[r * PP_ROW_WORDS + lane] = __ldg(si + lane); rowI[r * PP_ROW_WORDS + 32 + lane] = __ldg(si + 32 + lane);
        rowQ[r * PP_ROW_WORDS + lane] = __ldg(sq + lane); rowQ[r * PP_ROW_WORDS + 32 + lane] = __ldg(sq + 32 + lane);
      }
    }
    __syncthreads();
    int16_t *ri = reinterpret_cast<int16_t *>(rowI + lane * PP_ROW_WORDS), *rq = reinterpret_cast<int16_t *>(rowQ + lane * PP_ROW_WORDS);
    if (w == 0) {
      if (ch >= 0) pp_correct_block(ri, rq, s);
      sh_det[lane] = ch >= 0 && s.autod;
      sh_swap[lane] = s.swap;
    }
    __syncthreads();
    const bool det = sh_det[lane] != 0;
    if (__any_sync(0xFFFFFFFFu, det)) { /* same lanes, same flags in every warp: uniform over the CTA */
      if (det) {
        for (int i = w; i < 128; i += PP_W) {
          mine[(2 * i) * 32] = aux_q15_to_float(ri[i]);
          mine[(2 * i + 1) * 32] = aux_q15_to_float(rq[i]);
        }
      }
      __syncthreads();
      for (int st = 0; st < 7; st++) {
        if (det) pp_fft128_stage(mine, 32, c_fft_tw, st, w, PP_W);
        __syncthreads();
      }
      float pw[128 / PP_W];
      if (det) {
#pragma unroll
        for (int k = 0; k < 128 / PP_W; k++) pw[k] = pp_power(mine, 32, w + k * PP_W);
      }
      __syncthreads();
      if (det) {
#pragma unroll
        for (int k = 0; k < 128 / PP_W; k++) mine[(w + k * PP_W) * 32] = pw[k];
      }
      __syncthreads();
      if (w == 0 && det) pp_decide(mine, 32, s);
    }
    if (kRec && w == 0 && ch >= 0) { /* after pp_decide when detection ran in this block, after pp_correct_block otherwise */
      const size_t n = L.n_channels;
      int32_t *o = rec + (size_t)b * SDR_PP_BS_FIELDS * n + row;
      o[SDR_PP_BS_AUTO_DETECT * n] = s.autod; o[SDR_PP_BS_CORRECTION * n] = s.corr; o[SDR_PP_BS_FAILURE_COUNT * n] = s.fail;
      o[SDR_PP_BS_SUCCESS_COUNT * n] = s.succ; o[SDR_PP_BS_SAVED_SAMPLE * n] = s.saved; o[SDR_PP_BS_SWAP * n] = s.swap;
    }
    for (int r = w; r < 32; r += PP_W) {
      const int rr = __shfl_sync(0xFFFFFFFFu, row, r), sw = sh_swap[r];
      if (rr >= 0) {
        const uint32_t *a = (sw ? rowQ : rowI) + r * PP_ROW_WORDS, *c = (sw ? rowI : rowQ) + r * PP_ROW_WORDS;
        uint32_t *di = reinterpret_cast<uint32_t *>(L.oi + (size_t)rr * L.out_pitch + (size_t)b * 128);
        uint32_t *dq = reinterpret_cast<uint32_t *>(L.oq + (size_t)rr * L.out_pitch + (size_t)b * 128);
        di[lane] = a[lane]; di[32 + lane] = a[32 + lane];
        dq[lane] = c[lane]; dq[32 + lane] = c[32 + lane];
      }
    }
    __syncthreads();
  }
  if (w == 0 && ch >= 0) L.state[ch] = s;
}

/* ================================================================== grabber ==== */
/* AudioGrabberComplex256.cpp:50-72 over a whole call: the snapshot after the call is the last pair of blocks that completed,
 * its first half possibly carried over from the channel's previous call.  A channel's pair phase is its own (phase[ch] =
 * blocks it has processed, mod 2): calls on subsets of the channels leave the channels out of step with each other.
 * 64 threads per channel, all reading the channel's phase before thread 0 moves it on (a CTA barrier: 4 channels per CTA).
 * Thread j < 32 owns chunk j of the first half: the snapshot's first half and the carried half, which it reads (a pair
 * completed by the call's first block) and then overwrites (a pair left open at the end of the call) -- in place, one
 * thread per 16 bytes, so the carried halves of channels the call skips stay where they are.  Thread 32 + j writes chunk j
 * of the snapshot's second half. */
struct GrabLaunch {
  const int16_t *I, *Q; unsigned long long pitch;
  int16_t *half;                /* [n_channels][256]: first block of an incomplete pair, interleaved */
  int16_t *outb;                /* [n_channels][512] */
  uint8_t *phase, *valid;       /* [n_channels]: blocks processed mod 2, _dataBufferValid */
  const uint32_t *ids;          /* row -> channel; NULL: row = channel */
  uint32_t n_rows, n_blocks;
};

__device__ __forceinline__ int4 grab_interleave4(const int16_t *I, const int16_t *Q) { /* 4 samples of each rail -> re,im,re,im,... */
  const uint2 a = *reinterpret_cast<const uint2 *>(I), b = *reinterpret_cast<const uint2 *>(Q);
  int4 o;
  o.x = (int)__byte_perm(a.x, b.x, 0x5410); o.y = (int)__byte_perm(a.x, b.x, 0x7632);
  o.z = (int)__byte_perm(a.y, b.y, 0x5410); o.w = (int)__byte_perm(a.y, b.y, 0x7632);
  return o;
}

#define GRAB_THREADS 256
__global__ void __launch_bounds__(GRAB_THREADS) grab_update_kernel(const GrabLaunch L) {
  const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t r = idx >> 6, j = idx & 63;
  const bool live = r < L.n_rows;
  const uint32_t ch = live ? (L.ids ? __ldg(L.ids + r) : r) : 0;
  const int p = live ? (int)L.phase[ch] : 0;
  __syncthreads();
  if (!live) return;
  const int n = (int)L.n_blocks;
  const int16_t *ri = L.I + (size_t)r * L.pitch, *rq = L.Q + (size_t)r * L.pitch;
  const int bs = (p + n - 1) & 1 ? n - 1 : n - 2; /* last block of the call that completes a pair; < 0: none, the snapshot stays */
  const int s4 = (int)(j & 31) * 4;              /* first sample of the chunk within its block */
  int16_t *out = L.outb + (size_t)ch * 512 + 8 * j;
  if (j < 32) {
    int4 *carry = reinterpret_cast<int4 *>(L.half + (size_t)ch * 256 + 2 * s4);
    if (bs >= 1) *reinterpret_cast<int4 *>(out) = grab_interleave4(ri + (size_t)(bs - 1) * 128 + s4, rq + (size_t)(bs - 1) * 128 + s4);
    else if (bs == 0) *reinterpret_cast<int4 *>(out) = *carry;
    if ((p + n) & 1) *carry = grab_interleave4(ri + (size_t)(n - 1) * 128 + s4, rq + (size_t)(n - 1) * 128 + s4);
  } else if (bs >= 0) {
    *reinterpret_cast<int4 *>(out) = grab_interleave4(ri + (size_t)bs * 128 + s4, rq + (size_t)bs * 128 + s4);
  }
  if (j == 0) {
    L.phase[ch] = (uint8_t)((p + n) & 1);
    if (bs >= 0) L.valid[ch] = 1;
  }
}

/* ---- 256-point FFT + power, one warp per snapshot (the per-pair snapshots of a process call and the spectrum tap).
 * The operation network is the radix-2 decimation-in-frequency one the test suite's checker restates (aux_cfft256_forward), one
 * rounding per operation (-fmad=false), twiddles from c_fft_tw256, power re*re + im*im in natural bin order: only the data
 * movement differs.  A lane holds 8 complex points; point index bits b7..b0.  Three register layouts, one per group of
 * three stages, with a warp-local shared-memory transpose between them:
 *   L0: lane = b7..b3, register r = b2..b0 (idx = 8 lane + r)      load (16-byte rows), stages 2 and 1, power
 *   LA: lane = b4..b0, r = b7..b5 (idx = 32 r + lane)               stages 128, 64, 32
 *   LB: lane = (b7..b5, b1 b0), r = b4..b2                          stages 16, 8, 4
 * In L0 bin brev8(idx) = brev3(r) * 32 + brev5(lane): each register's power store covers one 128-byte line.
 * fft_swz: a word address with idx's low 5 bits XORed by G(b7..b5) = (x << 2) | (x >> 1), which makes the 32 lanes of every
 * layout's access hit 32 distinct banks. */
#define FFT_WARP_WORDS 512 /* re[256], im[256] */
__device__ __forceinline__ int fft_swz(int idx) { const int x = idx >> 5; return (idx & 0xE0) | ((idx & 31) ^ ((x << 2) | (x >> 1))); }

struct FftTw { /* the lane's twiddles of stages 128 .. 4 (stages 2 and 1 use warp-uniform entries) */
  float2 a128[4], a64[2], a32, b16[4], b8[2], b4;
};
__device__ __forceinline__ float2 fft_tw(int k) { return make_float2(c_fft_tw256[2 * k], c_fft_tw256[2 * k + 1]); }
__device__ __forceinline__ void fft_load_tw(FftTw &t, int l) {
#pragma unroll
  for (int r = 0; r < 4; r++) t.a128[r] = fft_tw(32 * r + l);     /* j = 32 r + l, step 1 */
#pragma unroll
  for (int r = 0; r < 2; r++) t.a64[r] = fft_tw(2 * (32 * r + l)); /* j = 32 (r & 1) + l, step 2 */
  t.a32 = fft_tw(4 * l);                                            /* j = l, step 4 */
#pragma unroll
  for (int r = 0; r < 4; r++) t.b16[r] = fft_tw(8 * (4 * r + (l & 3)));  /* j = 4 r + b1b0, step 8 */
#pragma unroll
  for (int r = 0; r < 2; r++) t.b8[r] = fft_tw(16 * (4 * r + (l & 3))); /* j = 4 (r & 1) + b1b0, step 16 */
  t.b4 = fft_tw(32 * (l & 3));                                            /* j = b1b0, step 32 */
}

/* aux_cfft256_forward's butterfly: a' = a + b, b' = (a - b) * w, each product and sum rounded on its own */
__device__ __forceinline__ void fft_bfly(float &ar, float &ai, float &br, float &bi, const float2 w) {
  const float tr = ar - br, ti = ai - bi;
  ar = ar + br;
  ai = ai + bi;
  const float p0 = tr * w.x, p1 = ti * w.y, p2 = tr * w.y, p3 = ti * w.x;
  br = p0 - p1;
  bi = p2 + p3;
}

/* registers of layout `from` -> shared memory -> registers of the next layout (idx_w(r), idx_r(r): the points written and read) */
#define FFT_TRANSPOSE(IDX_W, IDX_R)                                                          \
  do {                                                                                       \
    __syncwarp();                                                                            \
    _Pragma("unroll") for (int r = 0; r < 8; r++) { sr[fft_swz(IDX_W)] = xr[r]; si[fft_swz(IDX_W)] = xi[r]; } \
    __syncwarp();                                                                            \
    _Pragma("unroll") for (int r = 0; r < 8; r++) { xr[r] = sr[fft_swz(IDX_R)]; xi[r] = si[fft_swz(IDX_R)]; } \
  } while (0)

/* the bin of register r of lane l after fft256_pow: brev3(r) * 32 + brev5(l) */
__device__ __forceinline__ int fft_bin(int r, int l) { return (((r & 1) << 2) | (r & 2) | (r >> 2)) * 32 + (int)(__brev((unsigned)l) >> 27); }

/* w[i]: point 8 l + i as (re | im << 16), layout L0.  pw[r] <- the power of bin fft_bin(r, l).  sm: the warp's
 * FFT_WARP_WORDS words of shared memory. */
__device__ __forceinline__ void fft256_pow(const uint32_t w[8], float *sm, const FftTw &t, int l, float pw[8]) {
  float *sr = sm, *si = sm + 256;
  float xr[8], xi[8];
#pragma unroll
  for (int r = 0; r < 8; r++) { xr[r] = (float)(int16_t)(w[r] & 0xFFFFu); xi[r] = (float)((int)w[r] >> 16); }
  FFT_TRANSPOSE(8 * l + r, 32 * r + l); /* L0 -> LA */
#pragma unroll
  for (int r = 0; r < 4; r++) fft_bfly(xr[r], xi[r], xr[r + 4], xi[r + 4], t.a128[r]);
#pragma unroll
  for (int r = 0; r < 8; r++) if (!(r & 2)) fft_bfly(xr[r], xi[r], xr[r + 2], xi[r + 2], t.a64[r & 1]);
#pragma unroll
  for (int r = 0; r < 8; r += 2) fft_bfly(xr[r], xi[r], xr[r + 1], xi[r + 1], t.a32);
  FFT_TRANSPOSE(32 * r + l, 32 * (l >> 2) + 4 * r + (l & 3)); /* LA -> LB */
#pragma unroll
  for (int r = 0; r < 4; r++) fft_bfly(xr[r], xi[r], xr[r + 4], xi[r + 4], t.b16[r]);
#pragma unroll
  for (int r = 0; r < 8; r++) if (!(r & 2)) fft_bfly(xr[r], xi[r], xr[r + 2], xi[r + 2], t.b8[r & 1]);
#pragma unroll
  for (int r = 0; r < 8; r += 2) fft_bfly(xr[r], xi[r], xr[r + 1], xi[r + 1], t.b4);
  FFT_TRANSPOSE(32 * (l >> 2) + 4 * r + (l & 3), 8 * l + r); /* LB -> L0 */
#pragma unroll
  for (int r = 0; r < 8; r++) if (!(r & 2)) fft_bfly(xr[r], xi[r], xr[r + 2], xi[r + 2], fft_tw(64 * (r & 1))); /* j = b0, step 64 */
#pragma unroll
  for (int r = 0; r < 8; r += 2) fft_bfly(xr[r], xi[r], xr[r + 1], xi[r + 1], fft_tw(0));
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const float a = xr[r] * xr[r], b = xi[r] * xi[r];
    pw[r] = a + b;
  }
}

/* power[256] of the snapshot (natural bin order) to `out` */
__device__ __forceinline__ void fft256_power(const uint32_t w[8], float *sm, const FftTw &t, int l, float *out) {
  float pw[8];
  fft256_pow(w, sm, t, l, pw);
  const int col = (int)(__brev((unsigned)l) >> 27);
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const int row = ((r & 1) << 2) | (r & 2) | (r >> 2); /* brev3 */
    out[row * 32 + col] = pw[r];
  }
}

/* 8 samples of each rail (16-byte loads) -> 8 points (re | im << 16) */
__device__ __forceinline__ void grab_interleave8(const int16_t *I, const int16_t *Q, uint32_t w[8]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4 *>(I)), b = __ldg(reinterpret_cast<const uint4 *>(Q));
  const uint32_t ai[4] = {a.x, a.y, a.z, a.w}, bi[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 4; i++) { w[2 * i] = __byte_perm(ai[i], bi[i], 0x5410); w[2 * i + 1] = __byte_perm(ai[i], bi[i], 0x7632); }
}

/* lane l's 8 points of slot k of row r (channel ch, pair phase p before the call): the pair the call's block e = 2k + 1 - p
 * completes, blocks e - 1 and e, block -1 being the carried half.  Lanes 0-15 hold the first block, lanes 16-31 the second. */
__device__ __forceinline__ void grab_slot_points(const GrabLaunch &L, uint32_t r, uint32_t ch, int p, uint32_t k, int l, uint32_t w[8]) {
  const int e = 2 * (int)k + 1 - p, blk = l < 16 ? e - 1 : e, s8 = 8 * (l & 15);
  if (blk < 0) {
    const uint4 *c = reinterpret_cast<const uint4 *>(L.half + (size_t)ch * 256 + 2 * s8);
    const uint4 u = c[0], v = c[1];
    w[0] = u.x; w[1] = u.y; w[2] = u.z; w[3] = u.w; w[4] = v.x; w[5] = v.y; w[6] = v.z; w[7] = v.w;
  } else {
    const size_t off = (size_t)r * L.pitch + (size_t)blk * 128 + s8;
    grab_interleave8(L.I + off, L.Q + off, w);
  }
}

#define FFT_THREADS 256
/* Every snapshot a process call publishes (sdr_grabber_process_device_snapshots), launched before grab_update_kernel on the
 * call's stream: it only reads the grabber's state (pair phase, carried half).  Item = (row, slot), row-major over
 * n_rows x S, S = (n_blocks + 1) / 2; one warp per item, grid-stride.  Slot k of a row whose channel has pair phase p is the
 * pair the call's block e = 2k + 1 - p completes: blocks e - 1 and e, block -1 being the carried half; slots k >=
 * (p + n_blocks) / 2 do not exist and are not written.  Lane l holds points 8 l .. 8 l + 7: lanes 0-15 the first block, lanes
 * 16-31 the second. */
__global__ void __launch_bounds__(FFT_THREADS) grab_snapshots_kernel(const GrabLaunch L, int16_t *snaps, float *power) {
  __shared__ float sm[FFT_THREADS / 32][FFT_WARP_WORDS];
  const int l = threadIdx.x & 31, wib = threadIdx.x >> 5;
  FftTw t;
  if (power) fft_load_tw(t, l);
  const uint32_t S = (L.n_blocks + 1) / 2;
  const unsigned long long items = (unsigned long long)L.n_rows * S, nw = (unsigned long long)gridDim.x * (FFT_THREADS / 32);
  for (unsigned long long it = (unsigned long long)blockIdx.x * (FFT_THREADS / 32) + wib; it < items; it += nw) {
    const uint32_t r = (uint32_t)(it / S), k = (uint32_t)(it - (unsigned long long)r * S);
    const uint32_t ch = L.ids ? __ldg(L.ids + r) : r;
    const int p = (int)L.phase[ch];
    if (k >= (p + L.n_blocks) / 2) continue; /* uniform over the warp */
    uint32_t w[8];
    grab_slot_points(L, r, ch, p, k, l, w);
    if (snaps) {
      uint4 *d = reinterpret_cast<uint4 *>(snaps + it * 512 + 16 * l);
      d[0] = make_uint4(w[0], w[1], w[2], w[3]);
      d[1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
    if (power) fft256_power(w, sm[wib], t, l, power + it * 256);
  }
}

/* Averaged waterfall lines (sdr_grabber_process_device_waterfall), launched before grab_update_kernel on the call's stream:
 * it reads the pair phases and carried halves as grab_snapshots_kernel does and averages the same slots' power K at a time.
 * A channel holds h < K pairs summed in acc[sel] (st = h << 1 | sel).  Number the pairs v = h + k for the call's slot k,
 * v < h standing for the held sum: with C = (p + n_blocks) / 2 slots the row completes nl = (h + C) / K lines, line m
 * summing v = mK .. mK + K - 1 in order, one rounding per add, then one IEEE division by K per bin.  Item (row, m), m <= Lmax,
 * one warp each, grid-stride: m < nl writes line m to lines[r * line_pitch + first[r] + m]; m == nl with (h + C) % K != 0
 * sums the trailing partial into acc[sel ^ 1].  Line 0 (or, when nl == 0, the partial) reads acc[sel], so reader and
 * writer never share a buffer; wf_advance_kernel then flips sel and stores the new h for the listed rows only, because the
 * other channels' sums stay where they are.  Lane l accumulates bins fft_bin(0..7, l) in registers. */
struct WfLaunch {
  float *acc;                    /* [2][n_channels][256] */
  uint32_t *st;                  /* [n_channels]: pairs held << 1 | accumulator buffer */
  float *lines;                  /* [n_rows][line_pitch][256] */
  const uint32_t *first;         /* device [n_rows]: row r's first line slot, NULL: 0 */
  unsigned long long line_pitch; /* in lines */
  uint32_t n_channels, K, Lmax;
};
__global__ void __launch_bounds__(FFT_THREADS) grab_waterfall_kernel(const GrabLaunch L, const WfLaunch W) {
  __shared__ float sm[FFT_THREADS / 32][FFT_WARP_WORDS];
  const int l = threadIdx.x & 31, wib = threadIdx.x >> 5;
  FftTw t;
  fft_load_tw(t, l);
  /* opaque to the compiler from here: kept in registers, instead of reloaded in every FFT of the loop below from constant
   * memory at per-lane addresses, which serialises */
  float *tf = reinterpret_cast<float *>(&t);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(FftTw) / 4); i++) asm volatile("" : "+f"(tf[i]));
  const uint32_t per = W.Lmax + 1;
  const unsigned long long items = (unsigned long long)L.n_rows * per, nw = (unsigned long long)gridDim.x * (FFT_THREADS / 32);
  for (unsigned long long it = (unsigned long long)blockIdx.x * (FFT_THREADS / 32) + wib; it < items; it += nw) {
    const uint32_t r = (uint32_t)(it / per), m = (uint32_t)(it - (unsigned long long)r * per);
    const uint32_t ch = L.ids ? __ldg(L.ids + r) : r;
    const int p = (int)L.phase[ch];
    const uint32_t s = W.st[ch], h = s >> 1, sel = s & 1;
    const uint32_t T = h + (p + L.n_blocks) / 2, nl = T / W.K;
    if (m > nl || (m == nl && T % W.K == 0)) continue; /* uniform over the warp */
    uint32_t v = m * W.K;
    const uint32_t v1 = min(v + W.K, T);
    float acc[8];
    if (v < h) { /* line 0 (or the partial) continues the held sum */
      const float *a = W.acc + ((size_t)sel * W.n_channels + ch) * 256;
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j] = a[fft_bin(j, l)];
      v = h;
    } else {
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j] = 0.0f;
    }
    for (; v < v1; v++) {
      uint32_t w[8];
      float pw[8];
      grab_slot_points(L, r, ch, p, v - h, l, w);
      fft256_pow(w, sm[wib], t, l, pw);
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j] = acc[j] + pw[j];
    }
    if (m < nl) {
      float *o = W.lines + ((size_t)r * W.line_pitch + (W.first ? __ldg(W.first + r) : 0u) + m) * 256;
      const float k = (float)W.K;
#pragma unroll
      for (int j = 0; j < 8; j++) o[fft_bin(j, l)] = __fdiv_rn(acc[j], k);
    } else {
      float *a = W.acc + ((size_t)(sel ^ 1) * W.n_channels + ch) * 256;
#pragma unroll
      for (int j = 0; j < 8; j++) a[fft_bin(j, l)] = acc[j];
    }
  }
}

/* after grab_waterfall_kernel, before grab_update_kernel moves the phases on: the listed rows' new held count and buffer */
__global__ void wf_advance_kernel(const GrabLaunch L, uint32_t *st, uint32_t K) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= L.n_rows) return;
  const uint32_t ch = L.ids ? __ldg(L.ids + r) : r;
  const uint32_t s = st[ch];
  st[ch] = ((((s >> 1) + (L.phase[ch] + L.n_blocks) / 2) % K) << 1) | ((s & 1) ^ 1);
}

/* Spectrum tap on the snapshots (SURVEY 8f row 3: the panadapter that consumes grab(); sdr_grabber_spectrum[_device]): power
 * row i <- the 256-point forward complex FFT of channel channels[i]'s snapshot (NULL: i), (re, im) int16 pairs taken as
 * floats, power re^2 + im^2 per bin in natural bin order, on the warp core above.  valid != NULL (while some channels have no
 * snapshot yet): rows of those channels are not written.  One warp per row, grid-stride. */
__global__ void __launch_bounds__(FFT_THREADS) grab_spectrum_kernel(const int16_t *snap, const uint32_t *channels, const uint8_t *valid,
                                                                    uint32_t n, float *power) {
  __shared__ float sm[FFT_THREADS / 32][FFT_WARP_WORDS];
  const int l = threadIdx.x & 31, wib = threadIdx.x >> 5;
  FftTw t;
  fft_load_tw(t, l);
  for (uint32_t i = blockIdx.x * (FFT_THREADS / 32) + wib; i < n; i += gridDim.x * (FFT_THREADS / 32)) {
    const uint32_t ch = channels ? __ldg(channels + i) : i;
    if (valid && !valid[ch]) continue; /* uniform over the warp */
    const uint4 *s = reinterpret_cast<const uint4 *>(snap + (size_t)ch * 512 + 16 * l);
    const uint4 u = s[0], v = s[1];
    const uint32_t w[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
    fft256_power(w, sm[wib], t, l, power + (size_t)i * 256);
  }
}

/* ================================================================== host side ==== */
static thread_local std::string g_err;
static int fail(int code, const std::string &m) { g_err = m; return code; }
#define CK(call)                                                                                                    \
  do {                                                                                                              \
    cudaError_t e_ = (call);                                                                                        \
    if (e_ != cudaSuccess) return fail(SDR_AUX_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
  } while (0)

static int upload_tables() {
  float h[64], tw[128];
  memcpy(h, AUX_IQ_HILBERT, sizeof h);
  memcpy(tw, AUX_FFT_TW, sizeof tw);
  CK(cudaMemcpyToSymbol(c_iq_h, h, sizeof h));
  CK(cudaMemcpyToSymbol(c_fft_tw, tw, sizeof tw));
  float tw256[256];
  memcpy(tw256, AUX_FFT_TW256, sizeof tw256);
  CK(cudaMemcpyToSymbol(c_fft_tw256, tw256, sizeof tw256));
  return 0;
}

static int check_planes(const void *a, const void *b, const void *c, const void *d, size_t in_pitch, size_t out_pitch, uint32_t n_blocks) {
  if (!a || !c || !d || n_blocks == 0) return fail(SDR_AUX_EINVAL, "null plane or n_blocks == 0");
  if ((in_pitch & 7) || (out_pitch & 7) || in_pitch < (size_t)n_blocks * 128 || out_pitch < (size_t)n_blocks * 128)
    return fail(SDR_AUX_EINVAL, "pitch must be a multiple of 8 elements and >= 128*n_blocks");
  if (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c | (uintptr_t)d) & 15) return fail(SDR_AUX_EINVAL, "planes must be 16-byte aligned");
  if (c == a || c == b || d == a || d == b || c == d) return fail(SDR_AUX_EINVAL, "output planes must not alias the inputs or each other");
  return 0;
}

/* device staging for the *_process_host entry points */
struct Staging {
  int16_t *p[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t pitch = 0; uint32_t blocks = 0;
  int ensure(uint32_t n_channels, uint32_t n_blocks, int planes) {
    if (n_blocks <= blocks && p[planes - 1]) return 0;
    release();
    pitch = (size_t)n_blocks * 128;
    for (int i = 0; i < planes; i++)
      if (cudaMalloc(&p[i], pitch * n_channels * sizeof(int16_t)) != cudaSuccess) { release(); return fail(SDR_AUX_ENOMEM, "cudaMalloc(staging) failed"); }
    blocks = n_blocks;
    return 0;
  }
  void release() { for (auto &q : p) { if (q) cudaFree(q); q = nullptr; } blocks = 0; }
};

/* A subset call's id list: distinct ids below n, n_ids >= 1; NULL with n_ids == n is the call on every channel. */
static int check_ids(const uint32_t *ids, uint32_t n_ids, uint32_t n, std::vector<uint8_t> &mark) {
  if (!ids) return n_ids == n ? 0 : fail(SDR_AUX_EINVAL, "channel_ids == NULL needs n_ids == n_channels");
  if (n_ids == 0) return fail(SDR_AUX_EINVAL, "n_ids == 0");
  mark.resize(n, 0);
  uint32_t i = 0;
  for (; i < n_ids && ids[i] < n && !mark[ids[i]]; i++) mark[ids[i]] = 1;
  for (uint32_t k = 0; k < i; k++) mark[ids[k]] = 0;
  if (i == n_ids) return 0;
  return fail(SDR_AUX_EINVAL, ids[i] >= n ? "channel id out of range" : "channel id listed twice");
}

/* A handle's device copy of a subset call's id list, uploaded from a pinned host copy on the call's stream.  The host copy
 * is rewritten only once the previous upload has completed (`copied`), and the device copy only once the kernels of the
 * previous subset call, perhaps queued on another stream, have read it (`read`, waited on by the next call's stream). */
struct IdList {
  uint32_t *d = nullptr, *host = nullptr;
  cudaEvent_t copied = nullptr, read = nullptr;
  int init(uint32_t n) {
    if (cudaMalloc(&d, 4 * (size_t)n) != cudaSuccess || cudaMallocHost(&host, 4 * (size_t)n) != cudaSuccess) return fail(SDR_AUX_ENOMEM, "cudaMalloc(ids) failed");
    CK(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&read, cudaEventDisableTiming));
    return 0;
  }
  int upload(const uint32_t *ids, uint32_t n, cudaStream_t st) {
    CK(cudaEventSynchronize(copied));
    memcpy(host, ids, 4 * (size_t)n);
    CK(cudaStreamWaitEvent(st, read, 0));
    CK(cudaMemcpyAsync(d, host, 4 * (size_t)n, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(copied, st));
    return 0;
  }
  int done(cudaStream_t st) { CK(cudaEventRecord(read, st)); return 0; } /* after the call's last kernel that reads d */
  void release() {
    cudaFree(d); cudaFreeHost(host);
    if (copied) cudaEventDestroy(copied);
    if (read) cudaEventDestroy(read);
    d = host = nullptr; copied = read = nullptr;
  }
};

/* Checkpoint blobs: a tag and a version, then the channel's state (sdr_*_state_bytes() bytes each) */
enum : uint32_t { BLOB_PP = 0x50505358u, BLOB_IQ = 0x49515358u, BLOB_GRAB = 0x47525358u, BLOB_VERSION = 1u };
struct PpBlob { uint32_t tag, version; PpState s; };
struct IqBlob { uint32_t tag, version; float2 gains; int16_t hist[256]; };
struct GrabBlob { uint32_t tag, version; uint8_t phase, valid, fresh, pad[5]; int16_t half[256]; int16_t snap[512]; };

static int check_blob_ids(const uint32_t *ids, uint32_t n, uint32_t n_channels) {
  for (uint32_t i = 0; i < n; i++) if ((ids ? ids[i] : i) >= n_channels) return fail(SDR_AUX_EINVAL, "channel id out of range");
  return 0;
}
template <class B>
static int check_blobs(const void *blobs, uint32_t n, uint32_t tag) {
  for (uint32_t i = 0; i < n; i++) {
    B b;
    memcpy(&b, (const char *)blobs + i * sizeof(B), sizeof b);
    if (b.tag != tag || b.version != BLOB_VERSION) return fail(SDR_AUX_EINVAL, "import_state: not a state blob of this block and library version");
  }
  return 0;
}

/* ------------------------------------------------------------------ pre-processor ---- */
struct sdr_preproc {
  uint32_t n = 0; int device = 0;
  PpState *state = nullptr;
  uint32_t *list = nullptr, *count = nullptr;
  PpSetterCall *d_calls = nullptr; size_t d_calls_cap = 0;
  std::vector<PpSetterCall> pending;
  bool auto_possible = false; /* some channel may have its detector on */
  uint64_t launches = 0;
  Staging stg;
  int32_t *rec = nullptr; size_t rec_bytes = 0; /* device staging of the host form's block_status */
  IdList ids;
  std::vector<uint8_t> mark;
};

extern "C" int sdr_preproc_create(sdr_preproc_t **out, uint32_t n_channels, int device) {
  if (!out || n_channels == 0) return fail(SDR_AUX_EINVAL, "sdr_preproc_create: bad arguments");
  CK(cudaSetDevice(device));
  if (int rc = upload_tables()) return rc;
  CK(cudaFuncSetAttribute(pp_detect_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PP_DETECT_SMEM));
  CK(cudaFuncSetAttribute(pp_detect_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PP_DETECT_SMEM));
  CK(cudaFuncSetAttribute(pp_detect_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PP_DETECT_SMEM));
  CK(cudaFuncSetAttribute(pp_detect_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PP_DETECT_SMEM));
  sdr_preproc *h = new sdr_preproc();
  h->n = n_channels; h->device = device;
  if (cudaMalloc(&h->state, sizeof(PpState) * n_channels) != cudaSuccess || cudaMalloc(&h->list, 4 * (size_t)n_channels) != cudaSuccess ||
      cudaMalloc(&h->count, 4) != cudaSuccess) { sdr_preproc_destroy(h); return fail(SDR_AUX_ENOMEM, "cudaMalloc failed"); }
  if (int rc = h->ids.init(n_channels)) { sdr_preproc_destroy(h); return rc; }
  CK(cudaMemset(h->state, 0, sizeof(PpState) * n_channels)); /* PP.h:63-72 initialisers: everything 0 / false */
  *out = h;
  return 0;
}

extern "C" void sdr_preproc_destroy(sdr_preproc_t *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->state); cudaFree(h->list); cudaFree(h->count); cudaFree(h->d_calls); cudaFree(h->rec);
  h->stg.release();
  h->ids.release();
  delete h;
}

extern "C" int sdr_preproc_set(sdr_preproc_t *h, const uint32_t *channels, uint32_t n, uint32_t setter, int32_t arg) {
  if (!h) return fail(SDR_AUX_EINVAL, "null handle");
  if (setter < 1 || setter > 4) return fail(SDR_AUX_EINVAL, "unknown pre-processor setter " + std::to_string(setter));
  if (setter == SDR_PP_setI2SerrorCompensation && (arg < -1 || arg > 1)) return fail(SDR_AUX_EINVAL, "I2S compensation must be -1, 0 or +1");
  if (setter == SDR_PP_startAutoI2SerrorDetection) h->auto_possible = true;
  if (!channels) { h->pending.push_back({0xFFFFFFFFu, setter, arg, 0}); return 0; }
  for (uint32_t i = 0; i < n; i++) if (channels[i] >= h->n) return fail(SDR_AUX_EINVAL, "channel out of range");
  for (uint32_t i = 0; i < n; i++) h->pending.push_back({channels[i], setter, arg, 0});
  return 0;
}

static int pp_flush(sdr_preproc *h, cudaStream_t st) {
  if (h->pending.empty()) return 0;
  if (h->pending.size() > h->d_calls_cap) {
    cudaFree(h->d_calls); h->d_calls = nullptr;
    h->d_calls_cap = h->pending.size() * 2 + 64;
    if (cudaMalloc(&h->d_calls, sizeof(PpSetterCall) * h->d_calls_cap) != cudaSuccess) { h->d_calls_cap = 0; return fail(SDR_AUX_ENOMEM, "cudaMalloc(calls) failed"); }
  }
  /* pageable source: the copy is staged before the call returns, so the vector may be cleared right away */
  CK(cudaMemcpyAsync(h->d_calls, h->pending.data(), sizeof(PpSetterCall) * h->pending.size(), cudaMemcpyHostToDevice, st));
  pp_apply_kernel<<<(h->n + 255) / 256, 256, 0, st>>>(h->state, h->n, h->d_calls, (uint32_t)h->pending.size());
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(st)); /* d_calls may be reallocated by the next flush */
  h->pending.clear();
  h->launches++;
  return 0;
}

extern "C" int sdr_preproc_get_status(sdr_preproc_t *h, const uint32_t *channels, uint32_t n, sdr_preproc_status *out) {
  if (!h || !out) return fail(SDR_AUX_EINVAL, "null argument");
  CK(cudaSetDevice(h->device));
  if (int rc = pp_flush(h, 0)) return rc;
  CK(cudaDeviceSynchronize());
  const uint32_t cnt = channels ? n : h->n;
  for (uint32_t i = 0; i < cnt; i++) {
    const uint32_t c = channels ? channels[i] : i;
    if (c >= h->n) return fail(SDR_AUX_EINVAL, "channel out of range");
    PpState s;
    CK(cudaMemcpy(&s, h->state + c, sizeof s, cudaMemcpyDeviceToHost));
    out[i].auto_detect = s.autod; out[i].correction = s.corr; out[i].failure_count = s.fail;
    out[i].success_count = s.succ; out[i].saved_sample = s.saved; out[i].swap = s.swap;
  }
  return 0;
}

/* a process call's launches; ids: the device id list of a subset call (kList), else unused; rec: the call's per-block
 * records (device, NULL: none), written by the records instantiations of the finish and detect kernels */
template <bool kList>
static int pp_launch(sdr_preproc *h, const PpLaunch &L, const uint32_t *ids, int32_t *rec, cudaStream_t st) {
  const uint32_t n = L.n_channels, tb = (n + 255) / 256;
  const unsigned long long threads = (unsigned long long)n * L.n_blocks * 16;
  const unsigned sb = (unsigned)((threads + 255) / 256);
  if (h->auto_possible) {
    CK(cudaMemsetAsync(h->count, 0, 4, st));
    pp_list_kernel<kList><<<tb, 256, 0, st>>>(L, ids);
    h->launches++;
  }
  pp_static_kernel<kList><<<sb, 256, 0, st>>>(L, ids);
  if (rec) pp_finish_kernel<kList, true><<<(unsigned)(((unsigned long long)n * L.n_blocks + 255) / 256), 256, 0, st>>>(L, ids, rec);
  else pp_finish_kernel<kList, false><<<tb, 256, 0, st>>>(L, ids, nullptr);
  h->launches += 2;
  if (h->auto_possible) {
    if (rec) pp_detect_kernel<kList, true><<<(n + 31) / 32, 32 * PP_W, PP_DETECT_SMEM, st>>>(L, ids, rec);
    else pp_detect_kernel<kList, false><<<(n + 31) / 32, 32 * PP_W, PP_DETECT_SMEM, st>>>(L, ids, nullptr);
    h->launches++;
  }
  return 0;
}

static int check_block_status(const int32_t *block_status) {
  if ((uintptr_t)block_status & 15) return fail(SDR_AUX_EINVAL, "block_status must be 16-byte aligned");
  return 0;
}

extern "C" int sdr_preproc_process_device_status(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                                 size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
                                                 int32_t *block_status, void *cuda_stream) {
  if (!h) return fail(SDR_AUX_EINVAL, "null handle");
  if (int rc = check_ids(channel_ids, n_ids, h->n, h->mark)) return rc;
  if (!Q) return fail(SDR_AUX_EINVAL, "null plane");
  if (int rc = check_planes(I, Q, I_out, Q_out, in_pitch, out_pitch, n_blocks)) return rc;
  if (int rc = check_block_status(block_status)) return rc;
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (int rc = pp_flush(h, st)) return rc; /* setters of every channel, listed or not, in call order */
  PpLaunch L = {I, Q, I_out, Q_out, in_pitch, out_pitch, h->state, n_ids, n_blocks, h->list, h->count};
  if (channel_ids) {
    if (int rc = h->ids.upload(channel_ids, n_ids, st)) return rc;
    if (int rc = pp_launch<true>(h, L, h->ids.d, block_status, st)) return rc;
    if (int rc = h->ids.done(st)) return rc;
  } else if (int rc = pp_launch<false>(h, L, nullptr, block_status, st)) {
    return rc;
  }
  CK(cudaGetLastError());
  return 0;
}

extern "C" int sdr_preproc_process_device_subset(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                                 size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
                                                 void *cuda_stream) {
  return sdr_preproc_process_device_status(h, channel_ids, n_ids, I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks, nullptr, cuda_stream);
}

extern "C" int sdr_preproc_process_device(sdr_preproc_t *h, const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out,
                                          int16_t *Q_out, size_t out_pitch, uint32_t n_blocks, void *cuda_stream) {
  if (!h) return fail(SDR_AUX_EINVAL, "null handle");
  return sdr_preproc_process_device_status(h, nullptr, h->n, I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks, nullptr, cuda_stream);
}

/* host block_status: the records are staged in h->rec on the device and copied out before the call returns */
extern "C" int sdr_preproc_process_host_status(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                               size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks,
                                               int32_t *block_status) {
  if (!h || !I || !Q || !I_out || !Q_out || n_blocks == 0) return fail(SDR_AUX_EINVAL, "bad arguments");
  if (int rc = check_ids(channel_ids, n_ids, h->n, h->mark)) return rc;
  if (int rc = check_block_status(block_status)) return rc;
  CK(cudaSetDevice(h->device));
  if (int rc = h->stg.ensure(h->n, n_blocks, 4)) return rc;
  const size_t rec_bytes = block_status ? (size_t)n_blocks * SDR_PP_BS_FIELDS * n_ids * sizeof(int32_t) : 0;
  if (rec_bytes > h->rec_bytes) {
    cudaFree(h->rec); h->rec = nullptr; h->rec_bytes = 0;
    if (cudaMalloc(&h->rec, rec_bytes) != cudaSuccess) { h->rec = nullptr; return fail(SDR_AUX_ENOMEM, "cudaMalloc(block_status staging) failed"); }
    h->rec_bytes = rec_bytes;
  }
  const size_t w = (size_t)n_blocks * 128 * 2, dp = h->stg.pitch * 2;
  CK(cudaMemcpy2DAsync(h->stg.p[0], dp, I, in_pitch * 2, w, n_ids, cudaMemcpyHostToDevice, 0));
  CK(cudaMemcpy2DAsync(h->stg.p[1], dp, Q, in_pitch * 2, w, n_ids, cudaMemcpyHostToDevice, 0));
  if (int rc = sdr_preproc_process_device_status(h, channel_ids, n_ids, h->stg.p[0], h->stg.p[1], h->stg.pitch, h->stg.p[2], h->stg.p[3],
                                                 h->stg.pitch, n_blocks, block_status ? h->rec : nullptr, nullptr)) return rc;
  CK(cudaMemcpy2DAsync(I_out, out_pitch * 2, h->stg.p[2], dp, w, n_ids, cudaMemcpyDeviceToHost, 0));
  CK(cudaMemcpy2DAsync(Q_out, out_pitch * 2, h->stg.p[3], dp, w, n_ids, cudaMemcpyDeviceToHost, 0));
  if (block_status) CK(cudaMemcpyAsync(block_status, h->rec, rec_bytes, cudaMemcpyDeviceToHost, 0));
  CK(cudaStreamSynchronize(0));
  return 0;
}

extern "C" int sdr_preproc_process_host_subset(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                               size_t in_pitch, int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks) {
  return sdr_preproc_process_host_status(h, channel_ids, n_ids, I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks, nullptr);
}

extern "C" int sdr_preproc_process_host(sdr_preproc_t *h, const int16_t *I, const int16_t *Q, size_t in_pitch, int16_t *I_out,
                                        int16_t *Q_out, size_t out_pitch, uint32_t n_blocks) {
  if (!h) return fail(SDR_AUX_EINVAL, "bad arguments");
  return sdr_preproc_process_host_status(h, nullptr, h->n, I, Q, in_pitch, I_out, Q_out, out_pitch, n_blocks, nullptr);
}

extern "C" uint64_t sdr_preproc_launch_count(const sdr_preproc_t *h) { return h ? h->launches : 0; }

extern "C" size_t sdr_preproc_state_bytes(void) { return sizeof(PpBlob); }

extern "C" int sdr_preproc_export_state(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs) {
  if (!h || !blobs) return fail(SDR_AUX_EINVAL, "export_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, h->n)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  if (int rc = pp_flush(h, 0)) return rc; /* queued setters belong to the state being saved, as for get_status */
  CK(cudaDeviceSynchronize());
  std::vector<PpState> all(h->n);
  CK(cudaMemcpy(all.data(), h->state, sizeof(PpState) * h->n, cudaMemcpyDeviceToHost));
  for (uint32_t i = 0; i < n; i++) {
    const PpBlob b = {BLOB_PP, BLOB_VERSION, all[channel_ids ? channel_ids[i] : i]};
    memcpy((char *)blobs + i * sizeof b, &b, sizeof b);
  }
  return 0;
}

extern "C" int sdr_preproc_import_state(sdr_preproc_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs) {
  if (!h || !blobs) return fail(SDR_AUX_EINVAL, "import_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, h->n)) return rc;
  if (int rc = check_blobs<PpBlob>(blobs, n, BLOB_PP)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  if (int rc = pp_flush(h, 0)) return rc; /* earlier setters apply first; the blob then replaces the listed channels' state */
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    PpBlob b;
    memcpy(&b, (const char *)blobs + i * sizeof b, sizeof b);
    CK(cudaMemcpy(h->state + (channel_ids ? channel_ids[i] : i), &b.s, sizeof b.s, cudaMemcpyHostToDevice));
    if (b.s.autod) h->auto_possible = true; /* a running detector: pp_detect_kernel must be launched from now on */
  }
  return 0;
}

/* ------------------------------------------------------------------ I/Q generator ---- */
struct sdr_iqgen {
  uint32_t n = 0; int device = 0;
  int16_t *hist[2] = {nullptr, nullptr};
  int cur = 0; /* hist[cur] holds every channel's history; calls on every channel write the other buffer and flip it */
  float2 *gains = nullptr;
  std::vector<float2> h_gains;
  bool gains_dirty = true;
  uint64_t launches = 0;
  Staging stg;
  IdList ids;
  std::vector<uint8_t> mark;
};

extern "C" int sdr_iqgen_create(sdr_iqgen_t **out, uint32_t n_channels, int device) {
  if (!out || n_channels == 0) return fail(SDR_AUX_EINVAL, "sdr_iqgen_create: bad arguments");
  CK(cudaSetDevice(device));
  if (int rc = upload_tables()) return rc;
  sdr_iqgen *h = new sdr_iqgen();
  h->n = n_channels; h->device = device;
  h->h_gains.assign(n_channels, make_float2(1.0f, 1.0f)); /* IQ.h:72-73 */
  if (cudaMalloc(&h->hist[0], 512 * (size_t)n_channels) != cudaSuccess || cudaMalloc(&h->hist[1], 512 * (size_t)n_channels) != cudaSuccess ||
      cudaMalloc(&h->gains, sizeof(float2) * n_channels) != cudaSuccess) { sdr_iqgen_destroy(h); return fail(SDR_AUX_ENOMEM, "cudaMalloc failed"); }
  if (int rc = h->ids.init(n_channels)) { sdr_iqgen_destroy(h); return rc; }
  CK(cudaMemset(h->hist[0], 0, 512 * (size_t)n_channels)); /* the static buffers start at zero, IQ.cpp:37-38 */
  CK(cudaMemset(h->hist[1], 0, 512 * (size_t)n_channels));
  *out = h;
  return 0;
}

extern "C" void sdr_iqgen_destroy(sdr_iqgen_t *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->hist[0]); cudaFree(h->hist[1]); cudaFree(h->gains);
  h->stg.release();
  h->ids.release();
  delete h;
}

extern "C" int sdr_iqgen_set_gain_balance(sdr_iqgen_t *h, const uint32_t *channels, uint32_t n, float balance) {
  if (!h) return fail(SDR_AUX_EINVAL, "null handle");
  const float2 g = make_float2(balance, (float)(1.0 / (double)balance)); /* IQ.h:58-59 */
  if (!channels) { for (auto &x : h->h_gains) x = g; }
  else {
    for (uint32_t i = 0; i < n; i++) if (channels[i] >= h->n) return fail(SDR_AUX_EINVAL, "channel out of range");
    for (uint32_t i = 0; i < n; i++) h->h_gains[channels[i]] = g;
  }
  h->gains_dirty = true;
  return 0;
}

template <bool kList>
static void iq_launch(const IqLaunch &L, const uint32_t *ids, unsigned grid, cudaStream_t st) {
  iq_generate_kernel<kList><<<grid, IQ_THREADS, 0, st>>>(L, ids);
  iq_history_kernel<kList><<<(L.n_channels * 32 + 255) / 256, 256, 0, st>>>(L, ids);
}

extern "C" int sdr_iqgen_process_device_subset(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *X, size_t in_pitch,
                                               int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks, void *cuda_stream) {
  if (!h) return fail(SDR_AUX_EINVAL, "null handle");
  if (int rc = check_ids(channel_ids, n_ids, h->n, h->mark)) return rc;
  if (int rc = check_planes(X, nullptr, I_out, Q_out, in_pitch, out_pitch, n_blocks)) return rc;
  const uint32_t segs = (n_blocks * 128 + IQ_SEG - 1) / IQ_SEG;
  const unsigned long long grid = (unsigned long long)n_ids * segs;
  if (grid > 0x7FFFFFFFull) return fail(SDR_AUX_EINVAL, "too many channel-segments for one launch");
  CK(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  if (h->gains_dirty) {
    CK(cudaMemcpyAsync(h->gains, h->h_gains.data(), sizeof(float2) * h->n, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st)); /* pageable source may change after we return */
    h->gains_dirty = false;
  }
  IqLaunch L;
  L.x = X; L.oi = I_out; L.oq = Q_out; L.in_pitch = in_pitch; L.out_pitch = out_pitch;
  /* a call on every channel writes the new history to the other buffer and flips cur.  A subset call writes it in place:
   * the skipped channels' history stays in hist[cur].  Segment 0 of iq_generate_kernel, the only reader of the old
   * history, runs before the history kernel. */
  L.hist_in = h->hist[h->cur]; L.hist_out = h->hist[channel_ids ? h->cur : h->cur ^ 1]; L.gains = h->gains;
  L.n_samples = n_blocks * 128; L.n_channels = n_ids; L.segs = segs;
  if (channel_ids) {
    if (int rc = h->ids.upload(channel_ids, n_ids, st)) return rc;
    iq_launch<true>(L, h->ids.d, (unsigned)grid, st);
    if (int rc = h->ids.done(st)) return rc;
  } else {
    iq_launch<false>(L, nullptr, (unsigned)grid, st);
    h->cur ^= 1;
  }
  CK(cudaGetLastError());
  h->launches += 2;
  return 0;
}

extern "C" int sdr_iqgen_process_device(sdr_iqgen_t *h, const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out,
                                        size_t out_pitch, uint32_t n_blocks, void *cuda_stream) {
  if (!h) return fail(SDR_AUX_EINVAL, "null handle");
  return sdr_iqgen_process_device_subset(h, nullptr, h->n, X, in_pitch, I_out, Q_out, out_pitch, n_blocks, cuda_stream);
}

extern "C" int sdr_iqgen_process_host_subset(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *X, size_t in_pitch,
                                             int16_t *I_out, int16_t *Q_out, size_t out_pitch, uint32_t n_blocks) {
  if (!h || !X || !I_out || !Q_out || n_blocks == 0) return fail(SDR_AUX_EINVAL, "bad arguments");
  if (int rc = check_ids(channel_ids, n_ids, h->n, h->mark)) return rc;
  CK(cudaSetDevice(h->device));
  if (int rc = h->stg.ensure(h->n, n_blocks, 3)) return rc;
  const size_t w = (size_t)n_blocks * 128 * 2, dp = h->stg.pitch * 2;
  CK(cudaMemcpy2DAsync(h->stg.p[0], dp, X, in_pitch * 2, w, n_ids, cudaMemcpyHostToDevice, 0));
  if (int rc = sdr_iqgen_process_device_subset(h, channel_ids, n_ids, h->stg.p[0], h->stg.pitch, h->stg.p[1], h->stg.p[2], h->stg.pitch,
                                               n_blocks, nullptr)) return rc;
  CK(cudaMemcpy2DAsync(I_out, out_pitch * 2, h->stg.p[1], dp, w, n_ids, cudaMemcpyDeviceToHost, 0));
  CK(cudaMemcpy2DAsync(Q_out, out_pitch * 2, h->stg.p[2], dp, w, n_ids, cudaMemcpyDeviceToHost, 0));
  CK(cudaStreamSynchronize(0));
  return 0;
}

extern "C" int sdr_iqgen_process_host(sdr_iqgen_t *h, const int16_t *X, size_t in_pitch, int16_t *I_out, int16_t *Q_out,
                                      size_t out_pitch, uint32_t n_blocks) {
  if (!h) return fail(SDR_AUX_EINVAL, "bad arguments");
  return sdr_iqgen_process_host_subset(h, nullptr, h->n, X, in_pitch, I_out, Q_out, out_pitch, n_blocks);
}

extern "C" uint64_t sdr_iqgen_launch_count(const sdr_iqgen_t *h) { return h ? h->launches : 0; }

extern "C" size_t sdr_iqgen_state_bytes(void) { return sizeof(IqBlob); }

extern "C" int sdr_iqgen_export_state(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs) {
  if (!h || !blobs) return fail(SDR_AUX_EINVAL, "export_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, h->n)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    IqBlob b;
    b.tag = BLOB_IQ; b.version = BLOB_VERSION; b.gains = h->h_gains[c];
    CK(cudaMemcpy(b.hist, h->hist[h->cur] + (size_t)c * 256, sizeof b.hist, cudaMemcpyDeviceToHost));
    memcpy((char *)blobs + i * sizeof b, &b, sizeof b);
  }
  return 0;
}

extern "C" int sdr_iqgen_import_state(sdr_iqgen_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs) {
  if (!h || !blobs) return fail(SDR_AUX_EINVAL, "import_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, h->n)) return rc;
  if (int rc = check_blobs<IqBlob>(blobs, n, BLOB_IQ)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    IqBlob b;
    memcpy(&b, (const char *)blobs + i * sizeof b, sizeof b);
    CK(cudaMemcpy(h->hist[h->cur] + (size_t)c * 256, b.hist, sizeof b.hist, cudaMemcpyHostToDevice));
    h->h_gains[c] = b.gains;
  }
  h->gains_dirty = true;
  return 0;
}

/* ------------------------------------------------------------------ grabber ---- */
/* Each channel is one reference object with its own pair phase, _dataBufferValid and _newDataIsAvailable: calls on subsets
 * of the channels leave them in different states.  The device holds phase and validity for the kernels (grab_update_kernel
 * advances them); the host mirrors them for the readers. */
struct sdr_grabber {
  uint32_t n = 0; int device = 0;
  int16_t *half = nullptr, *outb = nullptr;
  uint8_t *d_phase = nullptr, *d_valid = nullptr;
  std::vector<uint8_t> phase, valid, fresh; /* blocks processed mod 2, _dataBufferValid, _newDataIsAvailable */
  uint32_t n_valid = 0;
  int fft_ctas = 1; /* resident CTAs of the warp-FFT kernels on the whole device: their grid */
  IdList ids;
  std::vector<uint8_t> mark;
};

extern "C" int sdr_grabber_create(sdr_grabber_t **out, uint32_t n_channels, int device) {
  if (!out || n_channels == 0) return fail(SDR_AUX_EINVAL, "sdr_grabber_create: bad arguments");
  CK(cudaSetDevice(device));
  if (int rc = upload_tables()) return rc; /* the spectrum tap's twiddles */
  sdr_grabber *h = new sdr_grabber();
  h->n = n_channels; h->device = device;
  h->phase.assign(n_channels, 0); h->valid.assign(n_channels, 0); h->fresh.assign(n_channels, 0);
  int sms = 0, per_sm = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, grab_snapshots_kernel, FFT_THREADS, 0) != cudaSuccess) {
    delete h; return fail(SDR_AUX_ECUDA, "cannot query the device's multiprocessors");
  }
  h->fft_ctas = std::max(1, sms * per_sm);
  if (cudaMalloc(&h->half, 512 * (size_t)n_channels) != cudaSuccess || cudaMalloc(&h->outb, 1024 * (size_t)n_channels) != cudaSuccess ||
      cudaMalloc(&h->d_phase, n_channels) != cudaSuccess || cudaMalloc(&h->d_valid, n_channels) != cudaSuccess) {
    sdr_grabber_destroy(h); return fail(SDR_AUX_ENOMEM, "cudaMalloc failed");
  }
  if (int rc = h->ids.init(n_channels)) { sdr_grabber_destroy(h); return rc; }
  CK(cudaMemset(h->half, 0, 512 * (size_t)n_channels));
  CK(cudaMemset(h->outb, 0, 1024 * (size_t)n_channels));
  CK(cudaMemset(h->d_phase, 0, n_channels));
  CK(cudaMemset(h->d_valid, 0, n_channels));
  *out = h;
  return 0;
}

extern "C" void sdr_grabber_destroy(sdr_grabber_t *h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->half); cudaFree(h->outb); cudaFree(h->d_phase); cudaFree(h->d_valid);
  h->ids.release();
  delete h;
}

/* grid of the warp-FFT kernels: at most one wave of resident CTAs, each warp then strides over the items */
static unsigned fft_grid(const sdr_grabber *h, unsigned long long items) {
  const unsigned long long need = (items + FFT_THREADS / 32 - 1) / (FFT_THREADS / 32), cap = (unsigned long long)h->fft_ctas;
  return (unsigned)std::max(1ull, std::min(need, cap));
}

/* ------------------------------------------------------------------ waterfall ---- */
/* Per channel: the pairs held (< K) and which of its two accumulator buffers holds their sum.  The device words st[] are
 * what the kernels read and advance; the host mirrors them (held, sel) for the line counts and the checkpoints, as the
 * grabber mirrors its pair phases. */
struct sdr_waterfall {
  uint32_t n = 0; int device = 0; uint32_t K = 1;
  float *acc = nullptr;   /* [2][n][256] */
  uint32_t *d_st = nullptr;
  std::vector<uint32_t> held;
  std::vector<uint8_t> sel;
  int ctas = 1;           /* resident CTAs of grab_waterfall_kernel on the whole device: its grid */
  IdList first;           /* device copy of a call's first line slots per row */
};

static uint32_t wf_lmax(uint32_t K, uint32_t n_blocks) { return (uint32_t)(((unsigned long long)K - 1 + (n_blocks + 1) / 2) / K); }

/* The grabber's process call with its optional outputs: snapshots / power per slot (grab_snapshots_kernel) and waterfall
 * lines (wf != NULL: grab_waterfall_kernel; counts then receive the lines per row, else the slots per row).  Every check
 * comes before anything is queued. */
static int grab_process(sdr_grabber *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q, size_t pitch,
                        uint32_t n_blocks, int16_t *snapshots, float *power, uint32_t *counts, sdr_waterfall *wf, float *lines,
                        size_t line_pitch, const uint32_t *first_line, cudaStream_t st) {
  if (!h || !I || !Q || n_blocks == 0) return fail(SDR_AUX_EINVAL, "bad arguments");
  if (int rc = check_ids(channel_ids, n_ids, h->n, h->mark)) return rc;
  if ((pitch & 7) || pitch < (size_t)n_blocks * 128 || (((uintptr_t)I | (uintptr_t)Q) & 15)) return fail(SDR_AUX_EINVAL, "planes must be 16-byte aligned, pitch a multiple of 8 and >= 128*n_blocks");
  if (((uintptr_t)snapshots | (uintptr_t)power) & 15) return fail(SDR_AUX_EINVAL, "snapshots and power must be 16-byte aligned");
  if (wf) {
    if (wf->n != h->n || wf->device != h->device) return fail(SDR_AUX_EINVAL, "the waterfall must have the grabber's device and channel count");
    if (!lines || ((uintptr_t)lines & 15)) return fail(SDR_AUX_EINVAL, "lines must be non-NULL and 16-byte aligned");
    for (uint32_t i = 0; i < n_ids; i++) {
      const uint32_t c = channel_ids ? channel_ids[i] : i;
      const unsigned long long nl = (wf->held[c] + (h->phase[c] + n_blocks) / 2) / wf->K;
      if ((first_line ? first_line[i] : 0ull) + nl > line_pitch) return fail(SDR_AUX_EINVAL, "a row's lines run past line_pitch");
    }
  }
  CK(cudaSetDevice(h->device));
  if (channel_ids) { if (int rc = h->ids.upload(channel_ids, n_ids, st)) return rc; }
  if (wf && first_line) { if (int rc = wf->first.upload(first_line, n_ids, st)) return rc; }
  GrabLaunch L = {I, Q, pitch, h->half, h->outb, h->d_phase, h->d_valid, channel_ids ? h->ids.d : nullptr, n_ids, n_blocks};
  if (snapshots || power) { /* reads the phases and carried halves before grab_update_kernel moves them on */
    grab_snapshots_kernel<<<fft_grid(h, (unsigned long long)n_ids * ((n_blocks + 1) / 2)), FFT_THREADS, 0, st>>>(L, snapshots, power);
    CK(cudaGetLastError());
  }
  if (wf) { /* the same, then the waterfall's words move on, then the phases */
    const uint32_t Lmax = wf_lmax(wf->K, n_blocks);
    const WfLaunch W = {wf->acc, wf->d_st, lines, first_line ? wf->first.d : nullptr, line_pitch, wf->n, wf->K, Lmax};
    const unsigned long long need = ((unsigned long long)n_ids * (Lmax + 1) + FFT_THREADS / 32 - 1) / (FFT_THREADS / 32);
    grab_waterfall_kernel<<<(unsigned)std::max(1ull, std::min(need, (unsigned long long)wf->ctas)), FFT_THREADS, 0, st>>>(L, W);
    CK(cudaGetLastError());
    wf_advance_kernel<<<(n_ids + 255) / 256, 256, 0, st>>>(L, wf->d_st, wf->K);
    CK(cudaGetLastError());
    if (first_line) { if (int rc = wf->first.done(st)) return rc; }
  }
  const unsigned long long threads = (unsigned long long)n_ids * 64;
  grab_update_kernel<<<(unsigned)((threads + GRAB_THREADS - 1) / GRAB_THREADS), GRAB_THREADS, 0, st>>>(L);
  CK(cudaGetLastError());
  if (channel_ids) { if (int rc = h->ids.done(st)) return rc; }
  for (uint32_t i = 0; i < n_ids; i++) { /* the host mirror of what the kernels do to phase, valid and the waterfall's words */
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    const bool completed = h->phase[c] + n_blocks >= 2; /* some block of this call completes a pair */
    const uint32_t slots = (h->phase[c] + n_blocks) / 2;
    if (wf) {
      const uint32_t T = wf->held[c] + slots;
      if (counts) counts[i] = T / wf->K;
      wf->held[c] = T % wf->K;
      wf->sel[c] ^= 1;
    } else if (counts) {
      counts[i] = slots;
    }
    h->phase[c] = (uint8_t)((h->phase[c] + n_blocks) & 1);
    if (completed) { h->n_valid += !h->valid[c]; h->valid[c] = 1; h->fresh[c] = 1; }
  }
  return 0;
}

extern "C" int sdr_grabber_process_device_snapshots(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I,
                                                    const int16_t *Q, size_t pitch, uint32_t n_blocks, int16_t *snapshots, float *power,
                                                    uint32_t *counts, void *cuda_stream) {
  return grab_process(h, channel_ids, n_ids, I, Q, pitch, n_blocks, snapshots, power, counts, nullptr, nullptr, 0, nullptr, (cudaStream_t)cuda_stream);
}

extern "C" int sdr_grabber_process_device_waterfall_at(sdr_grabber_t *gr, sdr_waterfall_t *wf, const uint32_t *channel_ids, uint32_t n_ids,
                                                       const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, float *lines,
                                                       size_t line_pitch, const uint32_t *first_line, uint32_t *counts, void *cuda_stream) {
  if (!wf) return fail(SDR_AUX_EINVAL, "null waterfall");
  return grab_process(gr, channel_ids, n_ids, I, Q, pitch, n_blocks, nullptr, nullptr, counts, wf, lines, line_pitch, first_line,
                      (cudaStream_t)cuda_stream);
}

extern "C" int sdr_grabber_process_device_waterfall(sdr_grabber_t *gr, sdr_waterfall_t *wf, const uint32_t *channel_ids, uint32_t n_ids,
                                                    const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, float *lines,
                                                    uint32_t *counts, void *cuda_stream) {
  if (!wf || n_blocks == 0) return fail(SDR_AUX_EINVAL, "bad arguments");
  return sdr_grabber_process_device_waterfall_at(gr, wf, channel_ids, n_ids, I, Q, pitch, n_blocks, lines, wf_lmax(wf->K, n_blocks), nullptr,
                                                 counts, cuda_stream);
}

extern "C" int sdr_waterfall_create(sdr_waterfall_t **out, uint32_t n_channels, int device, uint32_t K) {
  if (!out || n_channels == 0 || K == 0) return fail(SDR_AUX_EINVAL, "sdr_waterfall_create: bad arguments (n_channels >= 1, K >= 1)");
  CK(cudaSetDevice(device));
  if (int rc = upload_tables()) return rc;
  sdr_waterfall *w = new sdr_waterfall();
  w->n = n_channels; w->device = device; w->K = K;
  w->held.assign(n_channels, 0); w->sel.assign(n_channels, 0);
  int sms = 0, per_sm = 0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, grab_waterfall_kernel, FFT_THREADS, 0) != cudaSuccess) {
    delete w; return fail(SDR_AUX_ECUDA, "cannot query the device's multiprocessors");
  }
  w->ctas = std::max(1, sms * per_sm);
  if (cudaMalloc(&w->acc, 2 * 1024 * (size_t)n_channels) != cudaSuccess || cudaMalloc(&w->d_st, 4 * (size_t)n_channels) != cudaSuccess) {
    sdr_waterfall_destroy(w); return fail(SDR_AUX_ENOMEM, "cudaMalloc failed");
  }
  if (int rc = w->first.init(n_channels)) { sdr_waterfall_destroy(w); return rc; }
  CK(cudaMemset(w->acc, 0, 2 * 1024 * (size_t)n_channels));
  CK(cudaMemset(w->d_st, 0, 4 * (size_t)n_channels));
  *out = w;
  return 0;
}

extern "C" void sdr_waterfall_destroy(sdr_waterfall_t *w) {
  if (!w) return;
  cudaSetDevice(w->device);
  cudaFree(w->acc); cudaFree(w->d_st);
  w->first.release();
  delete w;
}

extern "C" int sdr_waterfall_get_info(const sdr_waterfall_t *w, uint32_t *n_channels, int *device, uint32_t *K) {
  if (!w || !n_channels || !device || !K) return fail(SDR_AUX_EINVAL, "get_info: bad arguments");
  *n_channels = w->n; *device = w->device; *K = w->K;
  return 0;
}

extern "C" int sdr_grabber_process_device_subset(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n_ids, const int16_t *I, const int16_t *Q,
                                                 size_t pitch, uint32_t n_blocks, void *cuda_stream) {
  return sdr_grabber_process_device_snapshots(h, channel_ids, n_ids, I, Q, pitch, n_blocks, nullptr, nullptr, nullptr, cuda_stream);
}

extern "C" int sdr_grabber_process_device(sdr_grabber_t *h, const int16_t *I, const int16_t *Q, size_t pitch, uint32_t n_blocks, void *cuda_stream) {
  if (!h) return fail(SDR_AUX_EINVAL, "bad arguments");
  return sdr_grabber_process_device_subset(h, nullptr, h->n, I, Q, pitch, n_blocks, cuda_stream);
}

extern "C" int sdr_grabber_new_data_available(sdr_grabber_t *h, uint32_t channel) {
  if (!h || channel >= h->n) return fail(SDR_AUX_EINVAL, "bad arguments");
  return h->fresh[channel];
}

/* Copies the snapshot rows of the channels that have one: row i of dst <- channel channels[i] (NULL: i), runs of
 * consecutive channels in one copy; rows of channels without a snapshot are not touched.  Returns the rows copied. */
static int copy_snapshot_rows(sdr_grabber *h, const uint32_t *channels, uint32_t cnt, int16_t *dst, cudaMemcpyKind kind, cudaStream_t st) {
  int written = 0;
  for (uint32_t i = 0; i < cnt;) {
    const uint32_t c = channels ? channels[i] : i;
    if (!h->valid[c]) { i++; continue; }
    uint32_t k = 1;
    while (i + k < cnt && (channels ? channels[i + k] : i + k) == c + k && h->valid[c + k]) k++;
    CK(cudaMemcpyAsync(dst + (size_t)i * 512, h->outb + (size_t)c * 512, 1024 * (size_t)k, kind, st));
    written += (int)k;
    i += k;
  }
  return written;
}

extern "C" int sdr_grabber_grab(sdr_grabber_t *h, const uint32_t *channels, uint32_t n, int16_t *dest) {
  if (!h || !dest) return fail(SDR_AUX_EINVAL, "bad arguments");
  const uint32_t cnt = channels ? n : h->n;
  for (uint32_t i = 0; i < cnt; i++) if ((channels ? channels[i] : i) >= h->n) return fail(SDR_AUX_EINVAL, "channel out of range");
  CK(cudaSetDevice(h->device));
  int written = 0;
  if (h->n_valid) { /* AudioGrabberComplex256.cpp:83-88, per channel */
    CK(cudaDeviceSynchronize());
    written = copy_snapshot_rows(h, channels, cnt, dest, cudaMemcpyDeviceToHost, 0);
    if (written < 0) return written;
    CK(cudaStreamSynchronize(0));
  }
  for (uint32_t i = 0; i < cnt; i++) h->fresh[channels ? channels[i] : i] = 0; /* AudioGrabberComplex256.cpp:90 */
  return written;
}

extern "C" int sdr_grabber_grab_device(sdr_grabber_t *h, int16_t *dest, void *cuda_stream) {
  if (!h || !dest) return fail(SDR_AUX_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->device));
  const int written = copy_snapshot_rows(h, nullptr, h->n, dest, cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream);
  if (written < 0) return written;
  std::fill(h->fresh.begin(), h->fresh.end(), (uint8_t)0);
  return written > 0 ? 1 : 0;
}

/* power[i*256 + k] = |FFT256(snapshot of channel i)|^2[k], device memory, for the listed channels (device array, NULL: all);
 * rows of channels without a snapshot are not written; returns 1 when some row was written, else 0.  Does not touch the
 * new-data flags. */
extern "C" int sdr_grabber_spectrum_device(sdr_grabber_t *h, const uint32_t *d_channels, uint32_t n, float *d_power, void *cuda_stream) {
  if (!h || !d_power) return fail(SDR_AUX_EINVAL, "bad arguments");
  CK(cudaSetDevice(h->device));
  if (!h->n_valid) return 0;
  const uint32_t cnt = d_channels ? n : h->n;
  if (cnt == 0) return 1;
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const bool every = h->n_valid == h->n;
  grab_spectrum_kernel<<<fft_grid(h, cnt), FFT_THREADS, 0, st>>>(h->outb, d_channels, every ? nullptr : h->d_valid, cnt, d_power);
  CK(cudaGetLastError());
  if (every) return 1;
  if (!d_channels) return 1;
  /* whether a listed channel has a snapshot: the list is in device memory */
  std::vector<uint32_t> ids(cnt);
  CK(cudaMemcpyAsync(ids.data(), d_channels, 4 * (size_t)cnt, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (uint32_t c : ids) if (c < h->n && h->valid[c]) return 1;
  return 0;
}

/* the same to HOST memory for the listed channels (NULL: all) */
extern "C" int sdr_grabber_spectrum(sdr_grabber_t *h, const uint32_t *channels, uint32_t n, float *power) {
  if (!h || !power) return fail(SDR_AUX_EINVAL, "bad arguments");
  const uint32_t cnt = channels ? n : h->n;
  for (uint32_t i = 0; i < cnt; i++) if ((channels ? channels[i] : i) >= h->n) return fail(SDR_AUX_EINVAL, "channel out of range");
  CK(cudaSetDevice(h->device));
  if (!h->n_valid) return 0;
  if (cnt == 0) return 0;
  /* the listed channels that have a snapshot, and their rows in `power` */
  std::vector<uint32_t> sel, rows;
  for (uint32_t i = 0; i < cnt; i++) {
    const uint32_t c = channels ? channels[i] : i;
    if (h->valid[c]) { sel.push_back(c); rows.push_back(i); }
  }
  if (sel.empty()) return 0;
  const bool every = !channels && sel.size() == cnt;
  const uint32_t m = (uint32_t)sel.size();
  uint32_t *d_ch = nullptr; float *d_p = nullptr;
  int rc = 0;
  do {
    if (cudaMalloc(&d_p, (size_t)m * 1024) != cudaSuccess) { rc = fail(SDR_AUX_ENOMEM, "cudaMalloc failed"); break; }
    if (!every) {
      if (cudaMalloc(&d_ch, (size_t)m * 4) != cudaSuccess) { rc = fail(SDR_AUX_ENOMEM, "cudaMalloc failed"); break; }
      if (cudaMemcpy(d_ch, sel.data(), (size_t)m * 4, cudaMemcpyHostToDevice) != cudaSuccess) { rc = fail(SDR_AUX_ECUDA, "copy failed"); break; }
    }
    grab_spectrum_kernel<<<fft_grid(h, m), FFT_THREADS>>>(h->outb, d_ch, nullptr, m, d_p);
    if (cudaGetLastError() != cudaSuccess) { rc = fail(SDR_AUX_ECUDA, "spectrum kernel failed"); break; }
    if (m == cnt) {
      if (cudaMemcpy(power, d_p, (size_t)m * 1024, cudaMemcpyDeviceToHost) != cudaSuccess) { rc = fail(SDR_AUX_ECUDA, "copy failed"); break; }
    } else {
      for (uint32_t k = 0; k < m && rc == 0; k++)
        if (cudaMemcpy(power + (size_t)rows[k] * 256, d_p + (size_t)k * 256, 1024, cudaMemcpyDeviceToHost) != cudaSuccess) rc = fail(SDR_AUX_ECUDA, "copy failed");
      if (rc) break;
    }
    rc = (int)m;
  } while (0);
  cudaFree(d_ch); cudaFree(d_p);
  return rc;
}

extern "C" size_t sdr_grabber_state_bytes(void) { return sizeof(GrabBlob); }

extern "C" int sdr_grabber_export_state(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n, void *blobs) {
  if (!h || !blobs) return fail(SDR_AUX_EINVAL, "export_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, h->n)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    GrabBlob b;
    memset(&b, 0, sizeof b);
    b.tag = BLOB_GRAB; b.version = BLOB_VERSION; b.phase = h->phase[c]; b.valid = h->valid[c]; b.fresh = h->fresh[c];
    CK(cudaMemcpy(b.half, h->half + (size_t)c * 256, sizeof b.half, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(b.snap, h->outb + (size_t)c * 512, sizeof b.snap, cudaMemcpyDeviceToHost));
    memcpy((char *)blobs + i * sizeof b, &b, sizeof b);
  }
  return 0;
}

extern "C" int sdr_grabber_import_state(sdr_grabber_t *h, const uint32_t *channel_ids, uint32_t n, const void *blobs) {
  if (!h || !blobs) return fail(SDR_AUX_EINVAL, "import_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, h->n)) return rc;
  if (int rc = check_blobs<GrabBlob>(blobs, n, BLOB_GRAB)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    GrabBlob b;
    memcpy(&b, (const char *)blobs + i * sizeof b, sizeof b);
    CK(cudaMemcpy(h->half + (size_t)c * 256, b.half, sizeof b.half, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->outb + (size_t)c * 512, b.snap, sizeof b.snap, cudaMemcpyHostToDevice));
    h->n_valid += (uint32_t)(b.valid != 0) - (uint32_t)h->valid[c];
    h->phase[c] = b.phase & 1; h->valid[c] = b.valid != 0; h->fresh[c] = b.fresh != 0;
  }
  CK(cudaMemcpy(h->d_phase, h->phase.data(), h->n, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->d_valid, h->valid.data(), h->n, cudaMemcpyHostToDevice));
  return 0;
}

/* the waterfall's blob: K (a sum of pairs is a part of a line only for the same K), the pairs held and their sum */
enum : uint32_t { BLOB_WF = 0x57465358u };
struct WfBlob { uint32_t tag, version, K, held; float acc[256]; };

extern "C" size_t sdr_waterfall_state_bytes(void) { return sizeof(WfBlob); }

extern "C" int sdr_waterfall_export_state(sdr_waterfall_t *w, const uint32_t *channel_ids, uint32_t n, void *blobs) {
  if (!w || !blobs) return fail(SDR_AUX_EINVAL, "export_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, w->n)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(w->device));
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    WfBlob b;
    b.tag = BLOB_WF; b.version = BLOB_VERSION; b.K = w->K; b.held = w->held[c];
    memset(b.acc, 0, sizeof b.acc); /* with no pair held the buffer is never read, and holds whatever sum it last received */
    if (b.held) CK(cudaMemcpy(b.acc, w->acc + ((size_t)w->sel[c] * w->n + c) * 256, sizeof b.acc, cudaMemcpyDeviceToHost));
    memcpy((char *)blobs + i * sizeof b, &b, sizeof b);
  }
  return 0;
}

extern "C" int sdr_waterfall_import_state(sdr_waterfall_t *w, const uint32_t *channel_ids, uint32_t n, const void *blobs) {
  if (!w || !blobs) return fail(SDR_AUX_EINVAL, "import_state: bad arguments");
  if (int rc = check_blob_ids(channel_ids, n, w->n)) return rc;
  if (int rc = check_blobs<WfBlob>(blobs, n, BLOB_WF)) return rc;
  for (uint32_t i = 0; i < n; i++) {
    WfBlob b;
    memcpy(&b, (const char *)blobs + i * sizeof b, sizeof b);
    if (b.K != w->K || b.held >= w->K) return fail(SDR_AUX_EINVAL, "import_state: the blob is of a waterfall with another K");
  }
  if (n == 0) return 0;
  CK(cudaSetDevice(w->device));
  CK(cudaDeviceSynchronize());
  for (uint32_t i = 0; i < n; i++) {
    const uint32_t c = channel_ids ? channel_ids[i] : i;
    WfBlob b;
    memcpy(&b, (const char *)blobs + i * sizeof b, sizeof b);
    CK(cudaMemcpy(w->acc + ((size_t)w->sel[c] * w->n + c) * 256, b.acc, sizeof b.acc, cudaMemcpyHostToDevice));
    w->held[c] = b.held;
  }
  std::vector<uint32_t> st(w->n);
  for (uint32_t c = 0; c < w->n; c++) st[c] = w->held[c] << 1 | w->sel[c];
  CK(cudaMemcpy(w->d_st, st.data(), 4 * (size_t)w->n, cudaMemcpyHostToDevice));
  return 0;
}

template <class H>
static int get_info(const H *h, uint32_t *n_channels, int *device) {
  if (!h || !n_channels || !device) return fail(SDR_AUX_EINVAL, "get_info: bad arguments");
  *n_channels = h->n; *device = h->device;
  return 0;
}
extern "C" int sdr_preproc_get_info(const sdr_preproc_t *h, uint32_t *n_channels, int *device) { return get_info(h, n_channels, device); }
extern "C" int sdr_iqgen_get_info(const sdr_iqgen_t *h, uint32_t *n_channels, int *device) { return get_info(h, n_channels, device); }
extern "C" int sdr_grabber_get_info(const sdr_grabber_t *h, uint32_t *n_channels, int *device) { return get_info(h, n_channels, device); }

extern "C" const char *sdr_aux_last_error(void) { return g_err.c_str(); }
extern "C" const char *sdr_aux_version(void) { return "audiosdr_b200 aux 0.1 (sm_100a)"; }
