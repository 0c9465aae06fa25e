// Shared helpers for the pygho_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pygho_b200.h"

namespace pgh {

void set_error(const char* fmt, ...);

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

inline int arg_error(const char* what) {
  set_error("bad argument: %s", what);
  return -1;
}

#define PGH_CUDA(expr)                                                   \
  do {                                                                   \
    cudaError_t _e = (expr);                                             \
    if (_e != cudaSuccess) {                                             \
      pgh::set_error("%s: %s", #expr, cudaGetErrorString(_e));           \
      return (int)_e;                                                    \
    }                                                                    \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline unsigned blocks_for(int64_t n, int per_block) {
  return (unsigned)((n + per_block - 1) / per_block);
}

constexpr int kSMs = 148;  // B200

extern int g_tune[16];  // run-time tuning knobs (pgh_set_tuning), defined in seg_gmr.cu

// Programmatic dependent launch (key 8, on by default): the launch is a programmatic edge of the
// stream / captured graph instead of a full serialisation, so that its launch latency hides under
// the predecessor's completion.  EVERY kernel launched through launch_pdl starts with pdl_enter():
// griddepcontrol.wait returns once the predecessor grids have completed and their writes are
// visible, i.e. before the kernel's first access to global memory.  No kernel triggers its
// dependents early (the trigger is implicit at grid completion): with griddepcontrol.
// launch_dependents at the top of every kernel the successor's CTAs sat on the SMs while the
// predecessor was still running -- a 7.4 us pooling kernel took 10.7 us in back-to-back replays and
// the training step gained less (128 graphs: 2.691 ms serialised, 2.623 ms early trigger, 2.608 ms
// implicit trigger; profiles/r2_pdl_trigger_ab.txt; -DPGH_PDL_EARLY_TRIGGER restores it).  Kernels
// of other libraries (cuBLAS, ATen) in between serialise as usual.
template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                       Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = g_tune[8] ? 1 : 0;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

#ifdef __CUDACC__
__device__ __forceinline__ void pdl_enter() {
#ifdef PGH_PDL_EARLY_TRIGGER
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#endif
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// activation of the MLP blocks (0 none, 1 SiLU, 2 ReLU); one definition so that the BatchNorm
// apply pass (fused_mlp.cu) and the eval GEMM epilogue (linear_stats.cu) round identically
template <int ACT>
__device__ __forceinline__ float act_fwd(float x) {
  if (ACT == 1) return x / (1.f + __expf(-x));
  if (ACT == 2) return fmaxf(x, 0.f);
  return x;
}
#endif

}  // namespace pgh
