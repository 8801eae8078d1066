// Kernels of the MLP value baseline (reference mjrl/mjrl/baselines/mlp_baseline.py: MLPBaseline._features / predict /
// fit, with the minibatch loop of mjrl/mjrl/utils/optimize_model.py: fit_data).
//
// The network is nn.Sequential(fc_0, ReLU, ..., fc_{L-1}) with widths dim = (S + 4,) + hidden + (1,).  Its parameters
// are one flat fp32 vector in model.parameters() order (W_0 [dim_1][dim_0], b_0, W_1, b_1, ...), which the Adam kernel
// of train.cuh updates in place.  Features are never stored for all rows: a row kernel forms them from the obs row and
// the int32 time index t of the row within its path,
//   x = [clip(obs, -10, 10) / 10, (t / 1000)^1 .. (t / 1000)^4]   (each in fp64, rounded to fp32 once; no constant column)
// Arithmetic is fp32 FMAs on the CUDA cores (a 64-row minibatch is far below a tensor-core tile); every sum runs in a
// fixed order, so the same inputs always give the same bits.
//
// One fit step is four launches, and nothing in it waits for the host (a captured graph of an epoch replays):
//   baseline_begin_kernel      minibatch cursor on the device; past the epoch's last minibatch the step is a no-op
//   baseline_rows_kernel<1>    per tile of minibatch rows: features, forward through every layer, dY = 2 (y_hat - y) / B,
//                              and the backward pass through the ReLU masks (all row-local); x, h_l and dZ_l go to the
//                              workspace
//   baseline_wgrad_kernel      every weight and bias gradient, summed over the B rows in row order (fp64 accumulators)
//   train_optim_batch_kernel   torch.optim.Adam, weight decay as the L2 term added to the gradient
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "train.cuh"

namespace simstep {

constexpr int kBlMaxLayers = 4;    // linear layers
constexpr int kBlMaxHidden = 256;
constexpr int kBlMaxObs = 512;
constexpr int kBlMaxBatch = 1024;
constexpr int kBlThreads = 512;
constexpr int kBlFitRows = 4;      // rows per CTA in a fit step: a 64-row minibatch spreads over 16 SMs
constexpr int kBlPredictRows = 8;

struct BlNet {
  int n_lin;                                            // linear layers
  int S;                                                // observation width; dim[0] = S + 4
  int dim[kBlMaxLayers + 1];                            // dim[n_lin] = 1
  long long w_off[kBlMaxLayers], b_off[kBlMaxLayers];  // offsets in the flat parameter vector
  long long P;                                          // parameters
};

// Fit-step workspace, one row per minibatch row: x [B][dim_0], h_l [B][dim_{l+1}] (hidden outputs after the ReLU),
// dz_l [B][dim_{l+1}] (gradient of the loss with respect to layer l's pre-activation; dz[n_lin - 1] is dY [B]).
struct BlWork {
  float* x;
  float* h[kBlMaxLayers - 1];
  float* dz[kBlMaxLayers];
};

// Minibatch cursor of the epoch being fitted (device memory, advanced by baseline_begin_kernel).
struct BlCtl {
  long long cursor;     // minibatches taken in this epoch
  long long n_batches;  // minibatches the epoch has: n // B - 1 (fit_data's count)
  long long row0;       // first permutation entry of the current minibatch
  int skip;             // the current step is past the epoch's end
};

// shared-memory floats of a tile of R rows: the input of every layer, plus (fit) the pre-activation gradients and
// the backward pass's partial sums
inline int bl_smem_floats(const BlNet& net, int R, bool fit) {
  int f = 0;
  for (int l = 0; l < net.n_lin; ++l) f += net.dim[l] + (fit ? net.dim[l + 1] : 0);
  return R * f + (fit ? R * kBlThreads : 0);  // fit: partial sums of the backward pass
}

__device__ inline float bl_feature(const float* __restrict__ obs_row, int S, int t, int c) {
  if (c < S) {
    const double v = fmin(fmax(static_cast<double>(obs_row[c]), -10.0), 10.0);
    return static_cast<float>(v / 10.0);
  }
  const double a = static_cast<double>(t) / 1000.0;
  double p = a;
  for (int j = S + 1; j <= c; ++j) p *= a;
  return static_cast<float>(p);
}

__device__ inline float bl_warp_sum(float v) {
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

__global__ void baseline_begin_kernel(BlCtl* c, OptimState* os, long long n_batches, int restart, int B, float beta1,
                                      float beta2) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (restart) c->cursor = 0;
  c->n_batches = n_batches;
  const int skip = c->cursor >= n_batches;
  c->skip = skip;
  os->skip = skip;
  if (skip) return;
  c->row0 = c->cursor * B;
  c->cursor += 1;
  optim_tick(os, beta1, beta2);
}

// FIT = false: out[i] = model(x_i) for rows i < n of obs / tidx.
// FIT = true: the B rows perm[row0 .. row0 + B) of the current minibatch, forward and backward into the workspace.
// Hidden layers: a warp per two output units, lanes over the units' inputs, each weight shared by the R rows of the
// tile; the output unit: one warp per row; the backward pass: a thread per (unit, slice of the next layer's units),
// all R rows at once.
template <bool FIT, int R>
__global__ void __launch_bounds__(kBlThreads)
baseline_rows_kernel(const BlNet net, const float* __restrict__ theta, const float* __restrict__ obs,
                     const int* __restrict__ tidx, long long n, const long long* __restrict__ perm,
                     const float* __restrict__ y, const BlCtl* __restrict__ ctl, int B, float* __restrict__ out,
                     BlWork wk) {
  extern __shared__ float sm[];
  long long row0 = 0, rows = n;
  if (FIT) {
    if (ctl->skip) return;
    row0 = ctl->row0;
    rows = B;
  }
  const int L = net.n_lin, S = net.S;
  int in_off[kBlMaxLayers], dz_off[kBlMaxLayers];  // tile of layer l's input rows / of dz_l
  int f = 0;
  for (int l = 0; l < L; ++l) { in_off[l] = f; f += R * net.dim[l]; }
  for (int l = 0; l < L; ++l) { dz_off[l] = f; f += R * net.dim[l + 1]; }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kWarps = kBlThreads / 32;
  const long long tiles = (rows + R - 1) / R;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long i0 = tile * R;
    const int nr = static_cast<int>(rows - i0 < R ? rows - i0 : R);
    const int d0 = net.dim[0];
    for (int idx = threadIdx.x; idx < R * d0; idx += kBlThreads) {
      const int r = idx / d0, c = idx - r * d0;
      float v = 0.f;
      if (r < nr) {
        const long long src = FIT ? perm[row0 + i0 + r] : i0 + r;
        v = bl_feature(obs + src * S, S, tidx[src], c);
        if (FIT) wk.x[(i0 + r) * d0 + c] = v;
      }
      sm[in_off[0] + idx] = v;
    }
    __syncthreads();
    for (int l = 0; l + 1 < L; ++l) {
      const int din = net.dim[l], dout = net.dim[l + 1];
      const float* __restrict__ W = theta + net.w_off[l];
      const float* __restrict__ bias = theta + net.b_off[l];
      const float* in = sm + in_off[l];
      float* h = sm + in_off[l + 1];
      // two units per warp and a few weight loads in flight: the weights stream from L2, latency bound otherwise
      for (int o = 2 * warp; o < dout; o += 2 * kWarps) {
        const bool two = o + 1 < dout;
        const float* __restrict__ w0 = W + static_cast<long long>(o) * din;
        const float* __restrict__ w1 = two ? w0 + din : w0;
        float a0[R], a1[R];
#pragma unroll
        for (int r = 0; r < R; ++r) a0[r] = a1[r] = 0.f;
#pragma unroll 4
        for (int k = lane; k < din; k += 32) {
          const float x0 = w0[k], x1 = w1[k];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            a0[r] = fmaf(x0, in[r * din + k], a0[r]);
            a1[r] = fmaf(x1, in[r * din + k], a1[r]);
          }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
          a0[r] = bl_warp_sum(a0[r]);
          a1[r] = bl_warp_sum(a1[r]);
        }
        if (lane < 2 && (lane == 0 || two)) {
          const int u = o + lane;
          const float b = bias[u];
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const float v = fmaxf((lane == 0 ? a0[r] : a1[r]) + b, 0.f);
            h[r * dout + u] = v;
            if (FIT && r < nr) wk.h[l][(i0 + r) * dout + u] = v;
          }
        }
      }
      __syncthreads();
    }
    {
      const int din = net.dim[L - 1];
      const float* __restrict__ W = theta + net.w_off[L - 1];
      const float b = theta[net.b_off[L - 1]];
      const float* in = sm + in_off[L - 1];
      for (int r = warp; r < nr; r += kWarps) {
        float acc = 0.f;
#pragma unroll 4
        for (int k = lane; k < din; k += 32) acc = fmaf(W[k], in[r * din + k], acc);
        acc = bl_warp_sum(acc);
        if (lane == 0) {
          const float v = acc + b;
          if (!FIT) {
            out[i0 + r] = v;
          } else {
            const float dy = (v - y[perm[row0 + i0 + r]]) * (2.f / static_cast<float>(B));  // MSELoss(mean) backward
            sm[dz_off[L - 1] + r] = dy;
            wk.dz[L - 1][i0 + r] = dy;
          }
        }
      }
    }
    if (FIT) {
      __syncthreads();
      // dz_l[r][k] = (sum_o dz_{l+1}[r][o] W_{l+1}[o][k]) [h_l[r][k] > 0]: thread (group q, k) sums the q-th slice of
      // o for all rows of the tile, the slices are added in order
      float* part = sm + dz_off[L - 1] + R;  // [kBlThreads][R] partial sums
      for (int l = L - 2; l >= 0; --l) {
        const int dk = net.dim[l + 1], dn = net.dim[l + 2];
        const float* __restrict__ W = theta + net.w_off[l + 1];
        const float* g = sm + dz_off[l + 1];
        const float* h = sm + in_off[l + 1];
        const int groups = kBlThreads / dk;   // dk <= kBlMaxHidden <= kBlThreads
        const int per = (dn + groups - 1) / groups;
        const int k = threadIdx.x % dk, q = threadIdx.x / dk;
        if (q < groups) {
          float acc[R];
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = 0.f;
          const int o1 = min(dn, (q + 1) * per);
#pragma unroll 8
          for (int o = q * per; o < o1; ++o) {
            const float w = W[static_cast<long long>(o) * dk + k];
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = fmaf(g[r * dn + o], w, acc[r]);
          }
#pragma unroll
          for (int r = 0; r < R; ++r) part[(q * R + r) * dk + k] = acc[r];
        }
        __syncthreads();
        for (int idx = threadIdx.x; idx < nr * dk; idx += kBlThreads) {
          const int r = idx / dk, kk = idx - r * dk;
          float acc = 0.f;
          for (int p = 0; p < groups; ++p) acc += part[(p * R + r) * dk + kk];
          const float v = h[idx] > 0.f ? acc : 0.f;
          sm[dz_off[l] + idx] = v;
          wk.dz[l][(i0 + r) * dk + kk] = v;
        }
        __syncthreads();
      }
    }
    __syncthreads();
  }
}

// The gradient of parameter p < net.P: dW_l[o][k] = sum_i dz_l[i][o] a_l[i][k] (a_0 = x, a_l = h_{l-1}), db_l[o] =
// sum_i dz_l[i][o]; rows i = 0 .. B-1 in order, fp64 accumulator.  Shared with the behaviour-cloning step (bc.cuh).
__device__ inline double bl_param_grad(const BlNet& net, int B, const BlWork& wk, long long p) {
  int l = 0;
  while (l + 1 < net.n_lin && p >= net.w_off[l + 1]) ++l;
  const int din = net.dim[l], dout = net.dim[l + 1];
  const float* __restrict__ dz = wk.dz[l];
  double acc = 0.0;
  if (p < net.b_off[l]) {
    const long long q = p - net.w_off[l];
    const int o = static_cast<int>(q / din), k = static_cast<int>(q - static_cast<long long>(o) * din);
    const float* __restrict__ a = l == 0 ? wk.x : wk.h[l - 1];
#pragma unroll 16
    for (int i = 0; i < B; ++i)
      acc = fma(static_cast<double>(dz[static_cast<long long>(i) * dout + o]), static_cast<double>(a[static_cast<long long>(i) * din + k]), acc);
  } else {
    const int o = static_cast<int>(p - net.b_off[l]);
#pragma unroll 16
    for (int i = 0; i < B; ++i) acc += static_cast<double>(dz[static_cast<long long>(i) * dout + o]);
  }
  return acc;
}

// grad[p] for every parameter p (bl_param_grad).
__global__ void __launch_bounds__(256)
baseline_wgrad_kernel(const BlNet net, const BlCtl* __restrict__ ctl, int B, BlWork wk, float* __restrict__ grad) {
  if (ctl->skip) return;
  for (long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; p < net.P;
       p += static_cast<long long>(gridDim.x) * blockDim.x)
    grad[p] = static_cast<float>(bl_param_grad(net, B, wk, p));
}

}  // namespace simstep
