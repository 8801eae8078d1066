// Launcher of the column-fused ensemble forward kernel (gemm_chain.cuh).  A translation unit of its own so that its
// (precision x activation) instantiations compile in parallel with api.cu.
#include <cuda.h>
#include <cuda_runtime.h>

#include "../../include/simstep.h"
#include "chain_launch.h"

namespace simstep {

namespace {

template <typename E, bool TANH>
cudaError_t launch_t(const ChainLaunch& cl, int sm_count, int device, cudaStream_t st) {
  static bool attr_set[64] = {};  // function attributes are per device
  auto kern = ensemble_chain_kernel<E, TANH>;
  constexpr size_t smem = GemmPlan<1, true>::smem_bytes();
  bool& done = attr_set[device % 64];
  if (!done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    done = true;
  }
  const int units = cl.args.m_tiles * cl.args.groups;
  if (units <= 0) return cudaSuccess;
  const int pairs = units < sm_count / 2 ? units : sm_count / 2;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(pairs * 2));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  return cudaLaunchKernelEx(&cfg, kern, cl.maps, cl.args);
}

template <typename E>
cudaError_t launch_a(bool tanh_act, const ChainLaunch& cl, int sm_count, int device, cudaStream_t st) {
  return tanh_act ? launch_t<E, true>(cl, sm_count, device, st) : launch_t<E, false>(cl, sm_count, device, st);
}

}  // namespace

cudaError_t launch_ensemble_chain(int prec, bool tanh_act, const ChainLaunch& cl, int sm_count, int device,
                                  cudaStream_t st) {
  switch (prec) {
    case SIMSTEP_PREC_TF32: return launch_a<ElemTF32>(tanh_act, cl, sm_count, device, st);
    case SIMSTEP_PREC_FP16: return launch_a<ElemF16>(tanh_act, cl, sm_count, device, st);
    case SIMSTEP_PREC_BF16: return launch_a<ElemBF16>(tanh_act, cl, sm_count, device, st);
  }
  return cudaErrorInvalidValue;
}

}  // namespace simstep
