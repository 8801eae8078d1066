// Interface between api.cu and chain.cu (the launcher of the column-fused ensemble forward kernel, gemm_chain.cuh).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include "gemm_chain.cuh"

namespace simstep {

struct ChainLaunch {
  ChainMaps maps;
  ChainArgs args;
};

// prec: SIMSTEP_PREC_*; tanh_act: hidden activation is tanh (ReLU otherwise).  Enqueues the launch on `st`
// (programmatic stream serialization): min(units, sm_count / 2) CTA pairs.  device: the calling thread's current device.
cudaError_t launch_ensemble_chain(int prec, bool tanh_act, const ChainLaunch& cl, int sm_count, int device,
                                  cudaStream_t st);

}  // namespace simstep
