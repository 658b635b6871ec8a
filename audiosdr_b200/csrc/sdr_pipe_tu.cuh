/* sdr_pipe_tu.cuh -- the receiver pipeline kernel for ONE tile length, compiled once per tile length.
 *
 * Included by sdr_pipe_t32.cu / sdr_pipe_t16.cu / sdr_pipe_t8.cu, each of which defines SDR_FIXED_T (tile length in samples, a
 * compile-time constant for everything in sdr_pipeline.cuh: loop bounds, tile strides and block arithmetic fold into the
 * instructions, measured 8 % faster than the same code with the tile length as a launch parameter) and SDR_TSUF (suffix of
 * the exported symbols).  The stages' code lives in a namespace of its own per tile length.
 */
#include <cuda_runtime.h>
#include <stdint.h>

#include "sdr_kernel.h"
#include "sdr_pipeline.cuh"

using namespace SDR_NS;

#define SDR_CAT2(a, b) a##b
#define SDR_CAT(a, b) SDR_CAT2(a, b)
#define SDR_SYM(name) SDR_CAT(name, SDR_TSUF)

__constant__ float2 c_hilbert2[64]; /* compact Hilbert half, H:757-774, every tap twice: the multiplicand pairs of the packed FIR */

/* ---- stage-to-stage hand-over (sdr_lay.h): one mbarrier per (stage, tile mod SDR_BAR_W), arrival count 1.  A stage
 * signals a finished tile with one arrive by lane 0 after re-converging the warp (the warp barrier orders the other
 * lanes' shared-memory and global writes before the arrive, whose release semantics publish them to the waiting
 * stages); a waiting stage polls the barrier's phase parity with mbarrier.try_wait (acquire), which suspends the warp in
 * hardware instead of spinning in the issue slots of the stages that share its scheduler. */
__device__ __forceinline__ void bar_init(uint32_t addr, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory"); }
__device__ __forceinline__ void bar_arrive(uint32_t addr) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory"); }
__device__ __forceinline__ bool bar_try(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bar_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
#if defined(SDR_WAIT_MODE) && SDR_WAIT_MODE == 1 /* experiment: non-blocking test + sleep instead of the suspending try_wait */
  for (;;) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    if (ok) break;
    __nanosleep(64);
  }
#elif defined(SDR_WAIT_MODE) && SDR_WAIT_MODE == 2 /* experiment: try_wait with an explicit suspend-time hint (ns) */
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(addr), "r"(parity), "r"(20000u) : "memory");
  } while (!ok);
#else
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
  } while (!ok);
#endif
}

/* CTA-wide barrier of warps that arrive from different instructions (every warp is a different stage): the unaligned
 * form after re-converging the warp.  Used once per launch, between the stages' state loads and their tile loops. */
__device__ __forceinline__ void cta_barrier() {
  __syncwarp();
  asm volatile("barrier.sync 0;" ::: "memory");
}

#ifdef SDR_LOCKSTEP
/* The lock-step schedule of the hand-over rules: at step s the stage with delay d works on tile s - d, one CTA-wide barrier
 * per step (the default: measured faster than the mbarrier hand-over below, DESIGN.md section 7). */
template <class Body>
__device__ __forceinline__ void pipeline_loop(const Ctx &x, int stage, Body body) {
  unsigned long long *prof = x.prof ? x.L->prof : nullptr; /* nullptr at compile time in the product kernel */
  const long long t_loaded = prof ? clock64() : 0;
  cta_barrier(); /* histories and tables are in shared memory */
  const uint32_t n = x.L->n_tiles;
  const int delay = x.Y->delay[stage];
  const uint32_t steps = n + (uint32_t)x.Y->dmax;
  const bool skip = prof && ((x.L->diag_skip >> stage) & 1u);
  long long busy = 0, waiting = 0;
  const long long t_begin = prof ? clock64() : 0;
  x.slots_reset();
#pragma unroll 1
  for (uint32_t s = 0; s < steps; s++) {
    const long long tau = (long long)s - delay;
    const long long t0 = prof ? clock64() : 0;
    if (tau >= 0 && tau < (long long)n) { if (!skip) body((uint32_t)tau); x.slots_advance(); }
    const long long t1 = prof ? clock64() : 0;
    cta_barrier();
    if (prof) { busy += t1 - t0; waiting += clock64() - t1; }
  }
  if (prof && (threadIdx.x & 31) == 0) {
    unsigned long long *row = prof + (size_t)blockIdx.x * SDR_PROF_SLOTS;
    row[stage] += (unsigned long long)busy;
    row[16 + stage] += (unsigned long long)waiting;
    if (x.Y->stage_of_warp[0] == stage) { row[14] += (unsigned long long)(clock64() - t_begin); row[15] += (unsigned long long)(t_loaded - x.t0); }
  }
}

/* A warp that runs several stages per step (merged plans, sdr_lay.h): `step(s)` works through the warp's program. */
template <class Step>
__device__ __forceinline__ void lockstep_loop(const Ctx &x, Step step) {
  cta_barrier();
  const uint32_t steps = x.L->n_tiles + (uint32_t)x.Y->dmax;
#pragma unroll 1
  for (uint32_t s = 0; s < steps; s++) { step(s); cta_barrier(); }
}
__device__ __forceinline__ bool tile_at(const Ctx &x, int stage, uint32_t s, uint32_t &tau) {
  const long long t = (long long)s - x.Y->delay[stage];
  tau = (uint32_t)t;
  return t >= 0 && t < (long long)x.L->n_tiles;
}

/* input and output of a group in one warp: both are short, memory-bound stages */
__device__ __forceinline__ void run_in_out(const Ctx &x, int lane) {
  RoleIn rin; RoleOut rout; rin.load(x, lane); rout.load(x, lane);
  Slots k_in, k_out; k_in.reset(); k_out.reset();
  lockstep_loop(x, [&](uint32_t s) {
    uint32_t t;
    if (tile_at(x, ST_IN, s, t)) { x.k = k_in; rin.step_a(x, lane, t); __syncwarp(); rin.step_b(x, lane, t); k_in.advance(x); }
    if (tile_at(x, ST_OUT, s, t)) { x.k = k_out; rout.step_a(x, lane, t); __syncwarp(); rout.step_b(x, lane, t); __syncwarp(); k_out.advance(x); }
  });
  rin.save(x, lane);
  x.k = k_out; rout.save(x, lane);
}

/* the envelope path of a SAM-only group in one warp (C:132-143): AM-phase NCO, image low-pass on both rails, magnitude.  It
 * computes only for blocks the PLL ended unlocked; the image filters' delay lines stay in the channel state between tiles
 * (loaded and stored around a tile that needs them), so the warp holds one cascade at a time. */
__device__ __forceinline__ void run_envelope_path(const Ctx &x, int lane) {
  RoleNco2 n2; RoleMag mg; n2.load(x, lane); mg.load(x, lane);
  x.k.reset();
  lockstep_loop(x, [&](uint32_t s) {
    uint32_t t;
    if (!tile_at(x, ST_NCO2, s, t)) return;
    if (__any_sync(0xffffffffu, n2.cid >= 0 && env_flag(x, lane, t) != 0)) {
      n2.step(x, lane, t);
      __syncwarp();
#pragma unroll 1
      for (int rail = 0; rail < 2; rail++) { RoleBiquad r; r.load(x, lane, 2, rail); r.step(x, lane, t); r.save(x); }
      __syncwarp();
      mg.step(x, lane, t);
    } else {
      mg.pass_locked(x, lane, t);
    }
    x.k.advance(x);
  });
  n2.save(x); mg.save(x);
}
#else
template <class Body>
__device__ __forceinline__ void pipeline_loop(const Ctx &x, int stage, Body body) {
  unsigned long long *prof = x.prof ? x.L->prof : nullptr; /* nullptr at compile time in the product kernel */
  const long long t_loaded = prof ? clock64() : 0;
  cta_barrier(); /* histories and tables are in shared memory */
  const uint32_t n = x.L->n_tiles, tpbm = (uint32_t)(x.tpb() - 1);
  const uint32_t bars = (uint32_t)__cvta_generic_to_shared(x.smem + x.o_bar());
  const bool skip = prof && ((x.L->diag_skip >> stage) & 1u);
  const uint32_t my_bar = bars + (uint32_t)x.Y->bar_of[stage] * (SDR_BAR_W * 8u);
  long long busy = 0, waiting = 0;
  const long long t_begin = prof ? clock64() : 0;
  x.slots_reset();
#pragma unroll 1
  for (uint32_t t = 0; t < n; t++) {
    const long long tw = prof ? clock64() : 0;
    { /* the stage's rules: all barriers are polled in one go (independent instructions), then only those still open */
      uint32_t addr[SDR_MAX_DEPS], par[SDR_MAX_DEPS], open_ = 0;
#pragma unroll
      for (int i = 0; i < SDR_MAX_DEPS; i++) {
        const SdrDep d = x.Y->deps[stage][i];
        const long long u = d.kind ? (long long)(t | tpbm) : (long long)t + d.k;
        addr[i] = bars + (uint32_t)(d.stage * SDR_BAR_W + ((uint32_t)u & (SDR_BAR_W - 1))) * 8u;
        par[i] = ((uint32_t)u / SDR_BAR_W) & 1u;
        if (d.stage >= 0 && u >= 0) open_ |= 1u << i;
      }
      while (open_) {
#pragma unroll
        for (int i = 0; i < SDR_MAX_DEPS; i++)
          if ((open_ >> i) & 1u) { if (bar_try(addr[i], par[i])) open_ &= ~(1u << i); }
      }
    }
    const long long t0 = prof ? clock64() : 0;
    if (!skip) body(t);
    __syncwarp();
    if ((threadIdx.x & 31) == 0) bar_arrive(my_bar + (t & (SDR_BAR_W - 1)) * 8u);
    x.slots_advance();
    if (prof) { const long long t1 = clock64(); waiting += t0 - tw; busy += t1 - t0; }
  }
  if (prof && (threadIdx.x & 31) == 0) {
    unsigned long long *row = prof + (size_t)blockIdx.x * SDR_PROF_SLOTS;
    row[stage] += (unsigned long long)busy;
    row[16 + stage] += (unsigned long long)waiting;
    if (x.Y->stage_of_warp[0] == stage) { row[14] += (unsigned long long)(clock64() - t_begin); row[15] += (unsigned long long)(t_loaded - x.t0); }
  }
}

#endif

/* One warp = one stage.  Stages common to both pipeline classes are instantiated once (ring offsets are run-time
 * values of the launch's plan) to keep the kernel's instruction footprint small: every warp runs different code, so
 * the hot loops of all stages have to share the instruction caches. */
__device__ __forceinline__ void run_stage(const Ctx &x, int stage, int lane) {
  const bool ssb = x.cls() == CLS_SSB;
  if (!x.Y->active[stage]) { pipeline_loop(x, stage, [&](uint32_t) {}); return; } /* a stage this bucket does not have: keeps step only */
#if defined(SDR_LOCKSTEP) && SDR_FIXED_T != 32
  if (x.Y->prog[threadIdx.x >> 5][1] != 0xFF) { /* merged plan: this warp runs several stages per step */
    if (stage == ST_IN) run_in_out(x, lane); else run_envelope_path(x, lane);
    return;
  }
#endif
  /* every 4-section cascade of the chain (IF rails, audio band-pass, AM image rails) runs through this one site */
  const bool is_if = stage == ST_IFI || stage == ST_IFQ, is_aud = stage == ST_AUD, is_img = !ssb && (stage == ST_IMGI || stage == ST_IMGQ);
  if (is_if || is_aud || is_img) {
    RoleBiquad r; r.load(x, lane, is_if ? 0 : (is_aud ? 1 : 2), is_if ? stage - ST_IFI : (is_img ? stage - ST_IMGI : 0));
    pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); });
    r.save(x);
    return;
  }
  switch (stage) {
    case ST_IN: {
      RoleIn r; r.load(x, lane);
      pipeline_loop(x, stage, [&](uint32_t t) { r.step_a(x, lane, t); __syncwarp(); r.step_b(x, lane, t); });
      r.save(x, lane);
    } break;
    case ST_NB: { RoleNb r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); r.save(x, lane); } break;
    case ST_ENVL: { RoleEnvl r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); } break;
    case ST_NBO: { RoleNbo r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); } break;
    case ST_AGC: { RoleAgc r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); r.save(x); } break;
    case ST_OUT: {
      RoleOut r; r.load(x, lane);
      pipeline_loop(x, stage, [&](uint32_t t) { r.step_a(x, lane, t); __syncwarp(); r.step_b(x, lane, t); __syncwarp(); });
      r.save(x, lane);
    } break;
    default:
      if (ssb) {
        if (stage == ST_NCO) {
          RoleNco r; r.load(x, lane);
          { /* does every active lane run the same oscillator? then one table per tile serves the whole group */
            const unsigned act = __ballot_sync(0xffffffffu, r.cid >= 0);
            const int leader = act ? __ffs(act) - 1 : 0;
            const uint32_t pb = __shfl_sync(0xffffffffu, f2u(r.phase), leader), ib = __shfl_sync(0xffffffffu, f2u(r.inc), leader);
            r.uniform = __all_sync(0xffffffffu, r.cid < 0 || (f2u(r.phase) == pb && f2u(r.inc) == ib)) != 0;
            if (r.uniform) { r.phase = u2f(pb); r.inc = u2f(ib); }
          }
          pipeline_loop(x, stage, [&](uint32_t t) {
            if (r.uniform) { r.table_step(x, lane); __syncwarp(); r.mix_step(x, lane, t); }
            else r.step(x, lane, t);
          });
          r.save(x);
        } else {
          const int sub = stage - ST_HIL0;
          RoleHilbert r; r.load(x, lane, sub);
          pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, reinterpret_cast<const float *>(c_hilbert2), lane, sub, t); });
          r.save(x, lane, sub);
        }
      } else {
        if (stage == ST_PLL) { RolePll r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); r.save(x); }
        else if (stage == ST_NCO2) { RoleNco2 r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); r.save(x); }
        else { RoleMag r; r.load(x, lane); pipeline_loop(x, stage, [&](uint32_t t) { r.step(x, lane, t); }); r.save(x); }
      }
      break;
  }
}

template <bool PROF, bool REC>
__device__ __forceinline__ void pipeline_cta(const SdrLaunch &L, unsigned char *smem) {
  Ctx x;
  x.L = &L;
  x.Y = &L.lay;
  x.G = &L.groups[blockIdx.x];
  x.smem = smem;
  x.gidx = (int)blockIdx.x;
  x.prof = PROF;
  x.rec = REC;
  x.t0 = PROF ? clock64() : 0;
  const int nthr = (int)blockDim.x;
  for (int i = threadIdx.x; i < 257; i += nthr) x.f(x.o_sine())[i] = L.tabs->sine[i];
  if (threadIdx.x < SDR_LANES) reinterpret_cast<int *>(smem + x.o_cid())[threadIdx.x] = x.G->row[threadIdx.x];
#ifndef SDR_LOCKSTEP
  {
    const uint32_t bars = (uint32_t)__cvta_generic_to_shared(smem + x.o_bar());
    for (int i = threadIdx.x; i < SDR_STAGES * SDR_BAR_W; i += nthr) bar_init(bars + 8u * (uint32_t)i, (uint32_t)x.Y->bar_count[i / SDR_BAR_W]);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
#endif
#ifdef SDR_BULK_IO
  if (threadIdx.x < 4) bulk_bar_init(smem + x.o_lut() + SDR_INBAR_OFF + 8 * threadIdx.x, SDR_LANES); /* input landing buffers: every lane of stage IN arrives */
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
  __syncthreads(); /* stage IN requests its first tile from load(), which needs the plane rows */
  for (int i = threadIdx.x; i < SDR_LUT_SLOTS * SDR_AGC_LUT_STRIDE; i += nthr) { /* the group's AGC tables */
    const int id = x.G->lut_ids[i / SDR_AGC_LUT_STRIDE];
    if (id >= 0) x.f(x.o_lut())[i] = L.agc_luts[(size_t)id * SDR_AGC_LUT_STRIDE + i % SDR_AGC_LUT_STRIDE];
  }
  /* Physical warp -> stage (SdrLay::stage_of_warp).  The warp scheduler of an SM sub-partition favours the HIGHER warp id
   * among eligible warps, and warp id % 4 picks the sub-partition, so the placement decides which stages compete for one
   * scheduler and who wins; the defaults for the 14-stage launches (sdr_types.h) were found by measurement
   * (tools/map_search.py). */
  const int phys = threadIdx.x >> 5, lane = threadIdx.x & 31;
  run_stage(x, (int)x.Y->stage_of_warp[phys], lane);
}

/* The product kernel, its twin that also writes per-block status records (launched when SdrLaunch::bstat is set), and the
 * diagnostics twin (per-stage busy / waiting counters, sub-phase timers, stage skipping; no records), launched only when the
 * handle was created with SDR_ROLE_PROFILE=1.  Keeping the counters and the record stores out of the product kernel is not
 * cosmetic: its stages are different instruction streams whose loops must share the instruction caches. */
/* register budget: the 32-sample plans run up to 14 warps, one CTA per SM; the shorter tiles exist for plans of at most 11
 * warps that share an SM two at a time (SDR_LB_THREADS / SDR_LB_BLOCKS are set by the sdr_pipe_t*.cu files) */
extern "C" __global__ void __launch_bounds__(SDR_LB_THREADS, SDR_LB_BLOCKS) SDR_SYM(sdr_pipeline_kernel)(const __grid_constant__ SdrLaunch L) {
  extern __shared__ __align__(16) unsigned char smem[];
  pipeline_cta<false, false>(L, smem);
}
extern "C" __global__ void __launch_bounds__(SDR_LB_THREADS, SDR_LB_BLOCKS) SDR_SYM(sdr_pipeline_rec_kernel)(const __grid_constant__ SdrLaunch L) {
  extern __shared__ __align__(16) unsigned char smem[];
  pipeline_cta<false, true>(L, smem);
}
extern "C" __global__ void __launch_bounds__(SDR_LB_THREADS, 1) SDR_SYM(sdr_pipeline_prof_kernel)(const __grid_constant__ SdrLaunch L) {
  extern __shared__ __align__(16) unsigned char smem[];
  pipeline_cta<true, false>(L, smem);
}

extern "C" int SDR_SYM(sdrk_setup_pipe)(const float *hilbert64) {
  float2 h2[64];
  for (int i = 0; i < 64; i++) h2[i] = make_float2(hilbert64[i], hilbert64[i]);
  cudaError_t e = cudaMemcpyToSymbol(c_hilbert2, h2, sizeof h2);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(SDR_SYM(sdr_pipeline_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(SDR_SYM(sdr_pipeline_rec_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(SDR_SYM(sdr_pipeline_prof_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
  if (e != cudaSuccess) return (int)e;
  /* launches that need less than half of an SM's shared memory are meant to share the SM: keep the carve-out at its maximum */
  e = cudaFuncSetAttribute(SDR_SYM(sdr_pipeline_kernel), cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(SDR_SYM(sdr_pipeline_rec_kernel), cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  if (e != cudaSuccess) return (int)e;
  e = cudaFuncSetAttribute(SDR_SYM(sdr_pipeline_prof_kernel), cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  return (int)e;
}

extern "C" int SDR_SYM(sdrk_launch_pipe)(const SdrLaunch *L, void *stream) {
  const int threads = L->lay.n_warps * 32, smem = L->lay.smem_bytes;
  if (L->prof) SDR_SYM(sdr_pipeline_prof_kernel)<<<L->n_groups, threads, smem, (cudaStream_t)stream>>>(*L);
  else if (L->bstat) SDR_SYM(sdr_pipeline_rec_kernel)<<<L->n_groups, threads, smem, (cudaStream_t)stream>>>(*L);
  else SDR_SYM(sdr_pipeline_kernel)<<<L->n_groups, threads, smem, (cudaStream_t)stream>>>(*L);
  return (int)cudaGetLastError();
}

/* resident CTAs per SM the hardware grants this launch configuration (diagnostics) */
extern "C" int SDR_SYM(sdrk_occupancy)(const SdrLaunch *L) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, SDR_SYM(sdr_pipeline_kernel), L->lay.n_warps * 32, (size_t)L->lay.smem_bytes) != cudaSuccess) return -1;
  return n;
}
