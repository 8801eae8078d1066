// Launcher of the column-fused ensemble forward kernel (gemm_chain.cuh).  A translation unit of its own so that its
// (precision x activation) instantiations compile in parallel with api.cu.
#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/simstep.h"
#include "chain_launch.h"
#include "launch.h"

namespace simstep {

cudaError_t launch_ensemble_chain(int prec, bool tanh_act, const ChainLaunch& cl, int sm_count, int device,
                                  cudaStream_t st) {
  constexpr size_t smem = GemmPlan<1, true>::smem_bytes();
  const int units = cl.args.m_tiles * cl.args.groups;
  const int pairs = units < sm_count / 2 ? units : sm_count / 2;
  cudaError_t e = cudaErrorInvalidValue;
  with_elem(prec, [&](auto elem) {
    auto kern = tanh_act ? ensemble_chain_kernel<decltype(elem), true> : ensemble_chain_kernel<decltype(elem), false>;
    e = raise_smem_limit(reinterpret_cast<const void*>(kern), device, smem);
    if (e == cudaSuccess && units > 0)
      e = launch_kernel(kern, dim3(unsigned(pairs * 2)), dim3(kGemmThreads), smem, st, kPdl | kPair, cl.maps, cl.args);
  });
  return e;
}

}  // namespace simstep
