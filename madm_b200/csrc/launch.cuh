// Programmatic dependent launch (PDL) plumbing.  A kernel launched through launch_k() with PDL on may become resident while its
// predecessor on the stream is still draining: its CTAs run their prologue (barrier init, TMEM allocation, tensor-map prefetch,
// index arithmetic) and then block in pdl_wait() until the predecessor has completed and its writes are visible.  Kernels call
// pdl_trigger() first so THEIR successor may be scheduled as soon as all of their own CTAs have started.
// Rules that keep this race-free: (1) every kernel launched through launch_k() executes pdl_wait() on every thread before its first
// global-memory access and before any early return; (2) kernels that are not PDL-aware are launched with <<<>>> and serialise as usual
// (griddepcontrol.* are no-ops without the launch attribute).
// The attribute is on inside training passes (PdlTrainScope) and off for inference.  A training pass at 2 images per GPU is ~1200
// eager launches of 5-40 us whose prologues are a visible fraction of each kernel: 64.0 -> 60.8 ms per training step (bench.py
// --config train, two runs each).  For inference it measured nothing (B200, bench.py, B = 8, CUDA-graph replay, 20 steps: 24.25 ->
// 24.17 ms per step for the base path, 50.36 -> 50.59 ms for the s0 variant): inside a graph the launch gaps are already ~1 us and
// the step runs at the board's power cap.
#pragma once
#include <cuda_runtime.h>

namespace madm {

inline bool& pdl_train_scope() {
  static thread_local bool on = false;
  return on;
}
struct PdlTrainScope {  // RAII: launches issued while one is alive carry the PDL attribute
  bool prev;
  PdlTrainScope() : prev(pdl_train_scope()) { pdl_train_scope() = true; }
  ~PdlTrainScope() { pdl_train_scope() = prev; }
};

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  if (pdl_train_scope()) {
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
  }
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

}  // namespace madm
