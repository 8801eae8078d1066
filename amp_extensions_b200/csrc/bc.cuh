// Behaviour cloning of the rollout policy (reference mjrl/mjrl/algos/behavior_cloning.py: BC.fit / mse_loss / mle_loss,
// over the Gaussian MLP of policy.cuh: mjrl/mjrl/policies/gaussian_mlp.py, mjrl/mjrl/utils/fc_network.py:42-55).
//
// The parameters being fitted are one flat fp32 vector in mjrl's get_param_values order (per layer W [out][in], b [out],
// then log_std [act]), which is the baseline's model.parameters() layout followed by log_std: the network part is
// described by a BlNet, and the baseline's gradient sum and the ensemble's Adam kernel are reused on it.  The
// transformations are read from the handle's policy tail (in_shift | in_div | out_scale | out_shift | std):
//     mu = (W_L act(... act(W_0 (obs - in_shift) / in_div + b_0) ...) + b_L) * out_scale + out_shift
//     MSE: loss = mean over B rows and act_dim columns of (mu - a)^2            (log_std is not in the graph)
//     MLE: loss = -mean_rows LL, LL = -1/2 sum_j z_j^2 - sum_j log_std_j - act_dim/2 log 2 pi, z = (a - mu) / exp(log_std)
// Arithmetic is fp32 FMAs on the CUDA cores; every sum runs in a fixed order, so the same inputs give the same bits.
//
// One fit step is four launches, and nothing in it waits for the host (a captured graph of an epoch replays):
//   baseline_begin_kernel      minibatch cursor on the device; past the epoch's int(n / B) minibatches a no-op
//   bc_rows_kernel<true>       per tile of minibatch rows: normalised input, forward through every layer, the output
//                              cotangent (and MLE's per-row log_std term), backward through tanh / relu; x, h_l, dz_l
//                              and the log_std terms go to the workspace
//   bc_grad_kernel             every weight, bias (and MLE log_std) gradient, summed over the B rows in row order in fp64
//   train_optim_batch_kernel   torch.optim.Adam; in MSE mode its count stops before log_std, which keeps its moments
// The full-data loss is bc_rows_kernel<false> (fp64 per-CTA partials {rows, loss sum, 0}) then moments_final_kernel.
// bc_commit_kernel writes the parameters into the policy (log_std clamped at min_log_std, as set_param_values does).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "baseline.cuh"
#include "npg.cuh"
#include "policy.cuh"
#include "train.cuh"

namespace simstep {

constexpr int kBcMaxBatch = 1024;
constexpr int kBcFitRows = 4;     // rows per CTA in a fit step: a 64-row minibatch spreads over 16 SMs
constexpr int kBcLossRows = 8;

enum BcLoss { kBcMse = 0, kBcMle = 1 };

struct BcNet {
  BlNet bl;          // the linear layers: dim = (obs_dim, hidden..., act_dim), flat offsets; bl.P = network parameters
  int act_dim;       // dim[n_lin]; log_std sits at flat index bl.P
  int tanh_act;      // 1 tanh, 0 relu
  int loss;          // BcLoss
};

// shared-memory floats of a tile of R rows: every layer's input and the output layer's pre-activation, then (fit) the
// pre-activation gradients of every layer and the backward pass's partial sums, or (loss) R fp64 row losses
inline int bc_smem_floats(const BcNet& net, int R, bool fit) {
  int f = 0;
  for (int l = 0; l <= net.bl.n_lin; ++l) f += R * net.bl.dim[l];
  if (fit) {
    for (int l = 0; l < net.bl.n_lin; ++l) f += R * net.bl.dim[l + 1];
    f += R * kBlThreads;
  } else {
    f = (f + 1) / 2 * 2 + 2 * R;
  }
  return f;
}

// FIT = false: the loss of rows 0 .. n-1, partial[blockIdx.x] = {rows, sum of row losses, 0} (fp64, row order).
// FIT = true: the B rows idx[row0 .. row0 + B) of the current minibatch, forward and backward into the workspace;
// lsg [B][act_dim] = d loss / d log_std per row (MLE).
// Layers: a warp per two output units, lanes over the units' inputs, each weight shared by the R rows of the tile (the
// baseline's scheme); the output stage: a thread per (row, action); the backward pass: a thread per (unit, slice of
// the next layer's units), all R rows at once, slices added in order.
template <bool FIT, int R>
__global__ void __launch_bounds__(kBlThreads)
bc_rows_kernel(const BcNet net, const float* __restrict__ theta, const float* __restrict__ tail,
               const float* __restrict__ obs, const float* __restrict__ act, long long n,
               const long long* __restrict__ idx, const BlCtl* __restrict__ ctl, int B, BlWork wk,
               float* __restrict__ lsg, double* __restrict__ partial) {
  extern __shared__ __align__(16) float sm_bc[];
  float* sm = sm_bc;
  long long row0 = 0, rows = n;
  if (FIT) {
    if (ctl->skip) return;
    row0 = ctl->row0;
    rows = B;
  }
  const int L = net.bl.n_lin, A = net.act_dim, D0 = net.bl.dim[0];
  const float* in_shift = tail;
  const float* in_div = tail + D0;
  const float* out_scale = in_div + D0;
  const float* out_shift = out_scale + A;
  const float* log_std = theta + net.bl.P;
  int in_off[kBlMaxLayers + 1], dz_off[kBlMaxLayers];  // tile of layer l's input rows (l = L: output pre-activation)
  int f = 0;
  for (int l = 0; l <= L; ++l) { in_off[l] = f; f += R * net.bl.dim[l]; }
  for (int l = 0; l < L; ++l) { dz_off[l] = f; f += R * net.bl.dim[l + 1]; }
  float* part = sm + f;                                                  // FIT: [kBlThreads][R] partial sums
  double* row_loss = reinterpret_cast<double*>(sm + (in_off[L] + R * A + 1) / 2 * 2);   // loss: [R]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kWarps = kBlThreads / 32;
  double cta_loss = 0.0;
  long long cta_rows = 0;
  const long long tiles = (rows + R - 1) / R;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long i0 = tile * R;
    const int nr = static_cast<int>(rows - i0 < R ? rows - i0 : R);
    for (int e = threadIdx.x; e < R * D0; e += kBlThreads) {
      const int r = e / D0, c = e - r * D0;
      float v = 0.f;
      if (r < nr) {
        const long long src = FIT ? idx[row0 + i0 + r] : i0 + r;
        v = (obs[src * D0 + c] - in_shift[c]) / in_div[c];
        if (FIT) wk.x[(i0 + r) * D0 + c] = v;
      }
      sm[in_off[0] + e] = v;
    }
    __syncthreads();
    for (int l = 0; l < L; ++l) {
      const bool last = l == L - 1;
      const int din = net.bl.dim[l], dout = net.bl.dim[l + 1];
      const float* __restrict__ W = theta + net.bl.w_off[l];
      const float* __restrict__ bias = theta + net.bl.b_off[l];
      const float* in = sm + in_off[l];
      float* h = sm + in_off[l + 1];
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
            float v = (lane == 0 ? a0[r] : a1[r]) + b;
            if (!last) {
              v = net.tanh_act ? tanhf(v) : fmaxf(v, 0.f);
              if (FIT && r < nr) wk.h[l][(i0 + r) * dout + u] = v;
            }
            h[r * dout + u] = v;
          }
        }
      }
      __syncthreads();
    }
    const float* pre = sm + in_off[L];
    if (!FIT) {
      const double c0 = 0.9189385332046727 * A;  // act_dim / 2 * log(2 pi)
      for (int r = threadIdx.x; r < nr; r += kBlThreads) {
        const long long src = i0 + r;
        double s = 0.0;
        for (int j = 0; j < A; ++j) {
          const double mu = static_cast<double>(fmaf(pre[r * A + j], out_scale[j], out_shift[j]));
          const double e = static_cast<double>(act[src * A + j]) - mu;
          if (net.loss == kBcMse) {
            s += e * e;
          } else {
            const double ls = static_cast<double>(log_std[j]);
            const double z = e / exp(ls);
            s += 0.5 * z * z + ls;
          }
        }
        row_loss[r] = net.loss == kBcMse ? s : s + c0;
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        for (int r = 0; r < nr; ++r) cta_loss += row_loss[r];
        cta_rows += nr;
      }
      __syncthreads();
      continue;
    }
    // output cotangent d loss / d pre-activation = d loss / d mu * out_scale
    {
      const float invB = 1.f / static_cast<float>(B);
      const float mse_scale = 2.f / (static_cast<float>(B) * static_cast<float>(A));
      float* dzL = sm + dz_off[L - 1];
      for (int e = threadIdx.x; e < R * A; e += kBlThreads) {
        const int r = e / A, j = e - r * A;
        float d = 0.f;
        if (r < nr) {
          const long long src = idx[row0 + i0 + r];
          const float mu = fmaf(pre[e], out_scale[j], out_shift[j]);
          const float a = act[src * A + j];
          if (net.loss == kBcMse) {
            d = (mu - a) * mse_scale * out_scale[j];
          } else {
            const float sd = expf(log_std[j]);
            const float z = (a - mu) / sd;
            d = -(z * invB / sd) * out_scale[j];
            lsg[(i0 + r) * A + j] = (1.f - z * z) * invB;
          }
          wk.dz[L - 1][(i0 + r) * A + j] = d;
        }
        dzL[e] = d;
      }
    }
    __syncthreads();
    // dz_l[r][k] = (sum_o dz_{l+1}[r][o] W_{l+1}[o][k]) act'(h_l[r][k]): thread (group q, k) sums the q-th slice of o
    // for all rows of the tile, the slices are added in order
    for (int l = L - 2; l >= 0; --l) {
      const int dk = net.bl.dim[l + 1], dn = net.bl.dim[l + 2];
      const float* __restrict__ W = theta + net.bl.w_off[l + 1];
      const float* g = sm + dz_off[l + 1];
      const float* h = sm + in_off[l + 1];
      const int groups = kBlThreads / dk;   // dk <= kPolicyMaxWidth < kBlThreads
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
      for (int e = threadIdx.x; e < nr * dk; e += kBlThreads) {
        const int r = e / dk, kk = e - r * dk;
        float acc = 0.f;
        for (int p = 0; p < groups; ++p) acc += part[(p * R + r) * dk + kk];
        const float hv = h[e];
        const float v = net.tanh_act ? acc * (1.f - hv * hv) : (hv > 0.f ? acc : 0.f);
        sm[dz_off[l] + e] = v;
        wk.dz[l][(i0 + r) * dk + kk] = v;
      }
      __syncthreads();
    }
    __syncthreads();
  }
  if (!FIT && threadIdx.x == 0) {
    partial[3 * blockIdx.x] = static_cast<double>(cta_rows);
    partial[3 * blockIdx.x + 1] = cta_loss;
    partial[3 * blockIdx.x + 2] = 0.0;
  }
}

// grad[p] for every network parameter (bl_param_grad) and, MLE, grad[P + j] = sum_i lsg[i][j] in row order (fp64).
__global__ void __launch_bounds__(256)
bc_grad_kernel(const BcNet net, const BlCtl* __restrict__ ctl, int B, BlWork wk, const float* __restrict__ lsg,
               float* __restrict__ grad) {
  if (ctl->skip) return;
  const long long total = net.bl.P + (net.loss == kBcMle ? net.act_dim : 0);
  for (long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; p < total;
       p += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (p < net.bl.P) {
      grad[p] = static_cast<float>(bl_param_grad(net.bl, B, wk, p));
    } else {
      const int j = static_cast<int>(p - net.bl.P);
      double acc = 0.0;
      for (int i = 0; i < B; ++i) acc += static_cast<double>(lsg[static_cast<long long>(i) * net.act_dim + j]);
      grad[p] = static_cast<float>(acc);
    }
  }
}

// The fitted parameters into the policy: log_std clamped at min_log_std in theta (MLP.set_param_values), every entry
// written to the pack / std tail with policy_store_flat, and to npg_theta (the NPG state's copy) when there is one.
__global__ void __launch_bounds__(256)
bc_commit_kernel(float* __restrict__ theta, int P, int ls0, float min_log_std, const int* __restrict__ pack_of,
                 float* __restrict__ pack, float* __restrict__ stdv, float* __restrict__ npg_theta) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x) {
    float t = theta[i];
    if (i >= ls0) {
      t = fmaxf(t, min_log_std);
      theta[i] = t;
    }
    if (npg_theta) npg_theta[i] = t;
    policy_store_flat(i, t, pack_of, ls0, pack, stdv);
  }
}

}  // namespace simstep
