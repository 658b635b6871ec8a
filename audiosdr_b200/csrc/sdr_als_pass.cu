/* sdr_als_pass.cu -- the ALS + output post-pass of a split ALS bucket (sdr_lay.h, lay_build_als).
 *
 * One warp per group (lane = channel), one CTA per warp, a quarter of an SM's shared memory or less: four groups per SM,
 * every one on an SM sub-partition scheduler of its own.  The warp is the chain's output stage (RoleOut: LMS line enhancer C:324-352, output
 * gain / mute / truncation C:160, staging rows, row-major stores) fed from the scratch plane the bucket's first launch wrote
 * instead of from the AGC stage's ring: tile t + 1 is requested (asynchronous copies) before tile t is swept, so its 4 KB are
 * in shared memory long before they are needed.  Same arithmetic, same state words as the single-launch form: a handle may
 * switch between the two from call to call. */
#include <cuda_runtime.h>
#include <stdint.h>

#define SDR_FIXED_T 32
#define SDR_RUNTIME_PLAN /* ring offsets and depths from the launch's plan (the 32-sample pipeline plan's constants do not apply) */
#define SDR_NS sdrk_als
#include "sdr_kernel.h"
#include "sdr_pipeline.cuh"

using namespace SDR_NS;

extern "C" __global__ void __launch_bounds__(32, 8) sdr_als_pass_kernel(const __grid_constant__ SdrLaunch L) {
  extern __shared__ __align__(16) unsigned char smem[];
  Ctx x;
  x.L = &L; x.Y = &L.lay; x.G = &L.groups[blockIdx.x]; x.smem = smem; x.gidx = (int)blockIdx.x; x.prof = false; x.rec = false; x.t0 = 0;
  const int lane = (int)threadIdx.x;
  reinterpret_cast<int *>(smem + x.o_cid())[lane] = x.G->row[lane];
  x.k.reset();
  RoleOut r; r.load(x, lane);
  const uint32_t n = L.n_tiles;
  RoleAlsIn::request(x, lane, 0, 0);
  cp_async_commit();
#pragma unroll 1
  for (uint32_t t = 0; t < n; t++) {
    cp_async_wait_pending(0);
    __syncwarp(); /* every lane's share of tile t is in; every lane is done with tile t - 1 */
    if (t + 1 < n) RoleAlsIn::request(x, lane, t + 1, Slots::next(x.k.c, x.nc()));
    cp_async_commit();
    if (x.Y->als_mirror) r.step_a<true>(x, lane, t); else r.step_a<false>(x, lane, t);
    __syncwarp();
    r.step_b(x, lane, t);
    __syncwarp();
    x.k.advance(x);
  }
  r.save(x, lane);
}

extern "C" int sdrk_setup_als_pass(void) {
  cudaError_t e = cudaFuncSetAttribute(sdr_als_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536);
  if (e != cudaSuccess) return (int)e;
  return (int)cudaFuncSetAttribute(sdr_als_pass_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}

extern "C" int sdrk_launch_als_pass(const SdrLaunch *L, void *stream) {
  if (L->n_groups == 0) return 0;
  sdr_als_pass_kernel<<<L->n_groups, 32, L->lay.smem_bytes, (cudaStream_t)stream>>>(*L);
  return (int)cudaGetLastError();
}

extern "C" int sdrk_occupancy_als_pass(const SdrLaunch *L) {
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, sdr_als_pass_kernel, 32, (size_t)L->lay.smem_bytes) != cudaSuccess) return -1;
  return n;
}
