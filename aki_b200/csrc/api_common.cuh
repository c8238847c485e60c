// Shared host-side helpers for the C-ABI entry points.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/aki_mma.h"

namespace aki {

void set_last_cuda_error(const char* msg);
// aki_mma_set_timing_events: one-shot pair of events recorded around the next tcgen05 attention kernel
void timing_hook_begin(cudaStream_t st);
void timing_hook_end(cudaStream_t st);

void count_launch();   // aki_mma_launch_count(): one tick per kernel this library enqueues

inline int check_launch() {
  count_launch();
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_last_cuda_error(cudaGetErrorString(e));
    return AKI_ERR_CUDA;
  }
  return AKI_OK;
}

// Programmatic dependent launch for the short kernels of a decode step (7 per layer, 5-35 us each): with the attribute a
// kernel's CTAs are scheduled as soon as every CTA of the previous kernel in the stream has passed its
// griddepcontrol.launch_dependents, and run up to their own griddepcontrol.wait -- which returns once the previous
// kernel has completed and its writes are visible.  Kernels launched this way execute pdl_prologue() before they touch
// memory another kernel may have written (weights, which no kernel writes, may be requested earlier).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }
template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// Same, with thread-block clusters of `cluster_x` CTAs along grid x.
template <typename... KArgs, typename... Args>
inline void launch_pdl_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                               unsigned cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster_x;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// (cols, rows) bf16 matrix with a row stride in elements -> TMA map of [32 x box_rows] SWIZZLE_64B boxes, the K-major
// UMMA operand layout (sm100_ptx.cuh sw64_offset); rows past the end load as zeros.  attn_fwd_sm100.cu.
int make_bf16_map_2d(CUtensorMap* m, const void* base, int cols, int rows, int64_t row_stride, int box_rows);

#define AKI_REQUIRE(cond, code) \
  do {                          \
    if (!(cond)) return (code); \
  } while (0)

}  // namespace aki
