// sf_probe.cuh — the kernels' measurement probes: a view inside sf_rollout_kernel that needs no profiler. Each probe is
// a build variant selected with a -D switch:
//   -DSF_BARRIER_TIMING  cycles the warps spend at the block barriers, in the stepping warp's stage preparation and in
//                        the sections of the step; read with sf_barrier_cycles (tools/gpu_barrier_timing.py)
//   -DSF_TIMELINE        globaltimer marks of warps 0 and 1 of every block; read with sf_timeline (tools/gpu_timeline.py,
//                        tools/gpu_block_cost.py)
// In the product build every macro below is a no-op. A probe adds code but no shared memory and no member to any
// structure, so a probe build measures the product's layout. Variants are built beside the product library
// (build.build(out=..., defs=...)) and loaded through SF_B200_LIB.
#pragma once
#include <cuda_runtime.h>

#include "../../include/sf_b200.h"

#ifdef SF_BARRIER_TIMING
// [0] drawing warps waiting for a prepared stage, [1] drawing-warp barriers, [2] warp 0 waiting for a free ring slot,
// [3..7] warp 0 preparing a stage (steps, memo state, round scans, stroke gathering, control words), [8..15] step sections
__device__ unsigned long long sf_bar_cycles[16];
__device__ __forceinline__ void sf_bar_add(int k, long long t0) { if ((threadIdx.x & 31) == 0) atomicAdd(&sf_bar_cycles[k], (unsigned long long)(clock64() - t0)); }
// SF_BT(k): the cycles since SF_BT_BEGIN() or the previous SF_BT go to counter k
#define SF_BT_BEGIN() long long tb_ = clock64()
#define SF_BT(k) do { sf_bar_add(k, tb_); tb_ = clock64(); } while (0)
// the same for the sections of the step, which only the lanes in `mask` (those that step an env) run
#define SF_ST_BEGIN(mask) unsigned stmask_ = (mask); long long ts_ = clock64()
#define SF_ST(k) do { __syncwarp(stmask_); sf_bar_add(k, ts_); ts_ = clock64(); } while (0)
#define SF_ST_RESTART(mask) do { stmask_ = (mask); ts_ = clock64(); } while (0)
// a use of the loaded word x (the branch is never taken), so that the section ends when the load has arrived
#define SF_ST_USE(x, y) do { if ((x) == 0x7fffffff) (y) = 0; } while (0)

extern "C" int sf_barrier_cycles(unsigned long long* h_out, int reset) {  // the 16 counters; zeroed after the read if reset
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(h_out, sf_bar_cycles, sizeof(unsigned long long) * 16);
  if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(sf_bar_cycles, z, sizeof(z)); }
  return SF_OK;
}
#else
#define SF_BT_BEGIN() ((void)0)
#define SF_BT(k) ((void)0)
#define SF_ST_BEGIN(mask) ((void)0)
#define SF_ST(k) ((void)0)
#define SF_ST_RESTART(mask) ((void)0)
#define SF_ST_USE(x, y) ((void)0)
#endif

#ifdef SF_TIMELINE
// tags: 1 kernel entry, 2 tables loaded, 3 first stage prepared, 4 arrival at a stage hand-over, 5 release from it, 7 end
#define SF_TL_BLOCKS 160
#define SF_TL_MAX 96
__device__ unsigned long long sf_tl[SF_TL_BLOCKS * 2 * SF_TL_MAX];  // (globaltimer ns << 8) | tag
__device__ int sf_tl_n[SF_TL_BLOCKS * 2];                            // marks of (block, warp) in the current launch
__device__ __forceinline__ void sf_tl_mark(int tag, bool first) {
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0 && warp < 2 && blockIdx.x < SF_TL_BLOCKS) {
    const int i = blockIdx.x * 2 + warp;
    const int k = first ? 0 : sf_tl_n[i];  // only this thread touches its counter during a launch
    sf_tl_n[i] = k + 1;
    if (k < SF_TL_MAX) {
      unsigned long long g;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
      sf_tl[i * SF_TL_MAX + k] = (g << 8) | (unsigned long long)tag;
    }
  }
}
#define SF_TL_START() sf_tl_mark(1, true)  // kernel entry: the first mark of a launch
#define SF_TL(tag) sf_tl_mark(tag, false)

extern "C" int sf_timeline(unsigned long long* h_out) {  // [160][2][SF_TL_MAX] marks, zeroed after the read; returns SF_TL_MAX
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(h_out, sf_tl, sizeof(unsigned long long) * SF_TL_BLOCKS * 2 * SF_TL_MAX);
  static unsigned long long z[SF_TL_BLOCKS * 2 * SF_TL_MAX];
  cudaMemcpyToSymbol(sf_tl, z, sizeof(z));
  return SF_TL_MAX;
}
#else
#define SF_TL_START() ((void)0)
#define SF_TL(tag) ((void)0)
#endif
