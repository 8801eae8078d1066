// How the library launches its kernels (api.cu and chain.cu): the dispatch from a run-time precision or member count
// to a kernel instantiation, the kernels' dynamic shared-memory limits, and the one launch function.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <type_traits>
#include <utility>

#include "../../include/simstep.h"
#include "gemm_tcgen05.cuh"

namespace simstep {

extern std::atomic<long long> g_launches;  // kernels launched by this process (simstep_launch_count)

// Calls f(ElemTF32{}), f(ElemF16{}) or f(ElemBF16{}) for SIMSTEP_PREC_TF32 / FP16 / BF16; false for any other value.
template <typename F>
bool with_elem(int prec, F&& f) {
  switch (prec) {
    case SIMSTEP_PREC_TF32: f(ElemTF32{}); return true;
    case SIMSTEP_PREC_FP16: f(ElemF16{}); return true;
    case SIMSTEP_PREC_BF16: f(ElemBF16{}); return true;
  }
  return false;
}

// Calls f(std::integral_constant<int, n>{}) for an ensemble of n in [1, 8] members; false for any other n.
template <typename F>
bool with_members(int n, F&& f) {
  switch (n) {
    case 1: f(std::integral_constant<int, 1>{}); return true;
    case 2: f(std::integral_constant<int, 2>{}); return true;
    case 3: f(std::integral_constant<int, 3>{}); return true;
    case 4: f(std::integral_constant<int, 4>{}); return true;
    case 5: f(std::integral_constant<int, 5>{}); return true;
    case 6: f(std::integral_constant<int, 6>{}); return true;
    case 7: f(std::integral_constant<int, 7>{}); return true;
    case 8: f(std::integral_constant<int, 8>{}); return true;
  }
  return false;
}

// Raises the dynamic shared-memory limit of `kern` on `device` (the calling thread's current device) to at least
// `bytes`.  The limit belongs to the kernel on the device, not to a handle, so it is never lowered: another handle's
// launches may need more.  Safe to call from several threads; once the limit is high enough it makes no runtime call.
cudaError_t raise_smem_limit(const void* kern, int device, size_t bytes);

enum LaunchFlags : unsigned {
  kPlain = 0,
  // programmatic stream serialization: the kernel may be scheduled while the stream's previous kernel drains.  Only for
  // kernels that begin with ptx::grid_dep_wait(); any other kernel would race with its predecessor.
  kPdl = 1,
  kPair = 2,  // clusters of two CTAs
};

// Every kernel launch of the library: counts the launch and returns its error.
template <typename... KArgs, typename... Args>
cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, unsigned flags,
                          Args&&... args) {
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (flags & kPdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n++].val.programmaticStreamSerializationAllowed = 1;
  }
  if (flags & kPair) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = 2;
    attr[n].val.clusterDim.y = 1;
    attr[n++].val.clusterDim.z = 1;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = n;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
  if (e == cudaSuccess) g_launches++;
  return e;
}

}  // namespace simstep
