// Launch side of the fast tile kernel (bd_step_tile.cuh), in its own translation unit so that its template
// instantiations compile in parallel with the generic kernel's (bd_kernels.cu).
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "bd_device.cuh"
#include "bd_params.h"
#include "bd_step_tile.cuh"

namespace bd {

template <int TASK, int A>
static cudaError_t launch_step_tile_t(const Params<float>& P, const LaunchSpec& ls, cudaStream_t st) {
  const int envs_per_tile = 4 * P.EW;
  const size_t smem = (size_t)envs_per_tile * P.M * P.D * 4;   // the [tile rows][D] observation tile and nothing else
  const bool vecrow = (A == 4) && (P.D % 4 == 0);
  const int aero = P.aero == 0 ? 0 : (P.aero == AERO_DW ? 1 : 2);
  void (*kern)(Params<float>);
  if (vecrow) kern = aero == 0 ? step_kernel_tile<TASK, A, (A == 4), 0> : (aero == 1 ? step_kernel_tile<TASK, A, (A == 4), 1> : step_kernel_tile<TASK, A, (A == 4), 2>);
  else kern = aero == 0 ? step_kernel_tile<TASK, A, false, 0> : (aero == 1 ? step_kernel_tile<TASK, A, false, 1> : step_kernel_tile<TASK, A, false, 2>);
  static size_t configured[6][64] = {{0}};
  size_t* const cfgd = configured[(vecrow ? 1 : 0) + 2 * aero];
  const int dv = ls.device & 63;
  if (smem > cfgd[dv]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cfgd[dv] = smem;
  }
  const int grid = P.grid_blocks > 0 ? P.grid_blocks : (P.N + envs_per_tile - 1) / envs_per_tile;
  // resident capacity of this kernel: with a grid at least that large, "every CTA of the previous launch has
  // started" implies "the launch before it has completed", so at most two launches are ever in flight
  static int per_sm[6][64] = {{0}};
  static size_t per_sm_smem[6][64] = {{0}};
  int& occ = per_sm[(vecrow ? 1 : 0) + 2 * aero][dv];
  if (occ == 0 || per_sm_smem[(vecrow ? 1 : 0) + 2 * aero][dv] != smem) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kBlock, smem) != cudaSuccess || occ < 1) occ = 1;
    per_sm_smem[(vecrow ? 1 : 0) + 2 * aero][dv] = smem;
  }
  Params<float> Q = P;
  // P.early_prefetch == 0: the launch right after bd_load_snapshot.  Its programmatic primary is the unpack kernel, which
  // wrote every ring plane, so nothing may be read before griddepcontrol.wait.  (With pipe_wait the kernel takes the
  // pipe_gate branch instead: the restore synchronised the stream, the finished-tile counter shows the previous step
  // complete, and every CTA executes griddepcontrol.wait before its first load.)
  Q.early_prefetch = (P.early_prefetch && ls.pdl && grid >= occ * ls.sm_count) ? 1 : 0;
  Q.pipe_wait = (P.pipeline && ls.pdl && grid >= occ * ls.sm_count) ? 1 : 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kBlock);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = ls.pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, Q);
}

// K steps in one launch (step_kernel_tile_many).  Plain stream order (no programmatic launch): the kernel starts when
// everything before it is complete and needs no epoch waits; it publishes epochs for the launches that follow.
template <int TASK, int A>
static cudaError_t launch_step_tile_many_t(const Params<float>& P, const ManySpan& span, const LaunchSpec& ls, cudaStream_t st) {
  const int envs_per_tile = 4 * P.EW;
  const size_t smem = 2 * (size_t)envs_per_tile * P.M * P.D * 4;
  const bool vecrow = (A == 4) && (P.D % 4 == 0);
  const int aero = P.aero == 0 ? 0 : (P.aero == AERO_DW ? 1 : 2);
  void (*kern)(Params<float>, ManySpan);
  if (vecrow) kern = aero == 0 ? step_kernel_tile_many<TASK, A, (A == 4), 0> : (aero == 1 ? step_kernel_tile_many<TASK, A, (A == 4), 1> : step_kernel_tile_many<TASK, A, (A == 4), 2>);
  else kern = aero == 0 ? step_kernel_tile_many<TASK, A, false, 0> : (aero == 1 ? step_kernel_tile_many<TASK, A, false, 1> : step_kernel_tile_many<TASK, A, false, 2>);
  static size_t configured[6][64] = {{0}};
  size_t* const cfgd = configured[(vecrow ? 1 : 0) + 2 * aero];
  const int dv = ls.device & 63;
  if (smem > cfgd[dv]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cfgd[dv] = smem;
  }
  const int grid = (P.N + envs_per_tile - 1) / envs_per_tile;
  kern<<<grid, kBlock, smem, st>>>(P, span);
  return cudaGetLastError();
}

template <int TASK>
static cudaError_t tile_many_a(int act_a, const Params<float>& P, const ManySpan& span, const LaunchSpec& ls, cudaStream_t st) {
  return act_a == 4 ? launch_step_tile_many_t<TASK, 4>(P, span, ls, st) : launch_step_tile_many_t<TASK, 1>(P, span, ls, st);
}

cudaError_t launch_step_tile_many(int task, int act_a, const Params<float>& P, int k, long long act_step, long long obs_step,
                                  long long out_step, const LaunchSpec& ls, cudaStream_t st) {
  ManySpan span;
  span.K = k; span.act_step = act_step; span.obs_step = obs_step; span.out_step = out_step;
  switch (task) {
    case TASK_HOVER: return tile_many_a<TASK_HOVER>(act_a, P, span, ls, st);
    case TASK_MULTIHOVER: return tile_many_a<TASK_MULTIHOVER>(act_a, P, span, ls, st);
    case TASK_SPIRAL: return tile_many_a<TASK_SPIRAL>(act_a, P, span, ls, st);
    default: return tile_many_a<TASK_SWARM>(act_a, P, span, ls, st);
  }
}

template <int TASK>
static cudaError_t tile_a(int act_a, const Params<float>& P, const LaunchSpec& ls, cudaStream_t st) {
  return act_a == 4 ? launch_step_tile_t<TASK, 4>(P, ls, st) : launch_step_tile_t<TASK, 1>(P, ls, st);
}

cudaError_t launch_step_tile(int task, int act_a, const Params<float>& P, const LaunchSpec& ls, cudaStream_t st) {
  switch (task) {
    case TASK_HOVER: return tile_a<TASK_HOVER>(act_a, P, ls, st);
    case TASK_MULTIHOVER: return tile_a<TASK_MULTIHOVER>(act_a, P, ls, st);
    case TASK_SPIRAL: return tile_a<TASK_SPIRAL>(act_a, P, ls, st);
    default: return tile_a<TASK_SWARM>(act_a, P, ls, st);
  }
}

}  // namespace bd
