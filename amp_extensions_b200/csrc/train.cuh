// Kernels around the GEMMs of the ensemble training step (reference milo/milo/dynamics.py:236-250,
// DynamicsModel.train_step: forward on normalised inputs, MSE against the normalised state difference, backward,
// optional gradient-norm clipping, SGD-Nesterov or Adam), all N members in one grouped pass, each on its own batch.
//
// The three GEMM families run on the tcgen05 kernel of gemm_tcgen05.cuh with tf32 operands and fp32 accumulation:
//   forward   h_l  = act(W_l [x | h_<l] + b_l)                       (as in the env step)
//   dgrad     dH_j = [dY_{j+1} | ... | dY_L] . BW_j                   K = output units of the layers that read h_j
//   wgrad     G_l  = dY_l^T . [x | h_<l]                              K = batch rows
// Both operands of that kernel are K-major, so the batch-reduction of wgrad reads TRANSPOSED copies of the
// activations and of the pre-activation gradients, and dgrad reads transposed slices of the weights (BW_j); the
// kernels below produce those copies, the loss gradient, the activation masks, the bias gradients, the gradient
// norm and the parameter update.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "elementwise.cuh"
#include "ptx.cuh"

namespace simstep {

// x rows of the training batch: member g's rows sit at [g * Bp, g * Bp + B), the rest of its tile is zero.
//   x[g*Bp + r] = [(s - mean_s)/scale_s ; (a - mean_a)/scale_a ; 0...]   (dynamics.py:225-230)
__global__ void train_prep_kernel(const float* __restrict__ state, const float* __restrict__ action, int S, int A,
                                  int XP, int B, int Bp, int n_members, const float* __restrict__ tf,
                                  float* __restrict__ x) {
  const long long total = static_cast<long long>(n_members) * Bp * XP;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int col = static_cast<int>(idx % XP);
    const long long row = idx / XP;
    const int r = static_cast<int>(row % Bp);
    const int g = static_cast<int>(row / Bp);
    float v = 0.f;
    if (r < B) {
      const long long src = static_cast<long long>(g) * B + r;
      if (col < S) {
        v = state[src * S + col];
        if (tf) v = (v - tf[col]) / tf[S + col];
      } else if (col < S + A) {
        v = action[src * A + col - S];
        if (tf) v = (v - tf[2 * S + col - S]) / tf[2 * S + A + col - S];
      }
    }
    x[idx] = ptx::round_tf32(v);
  }
}

constexpr int kTrainPartials = 256;  // partial sums per member and region (deterministic two-pass reductions)

// MSE loss and its gradient with respect to the final layer's output (dynamics.py:241-246):
//   target = ((s' - s) - mean_d) / scale_d,  e = pred - target,  loss_g = mean_{r<B, c<S} e^2,
//   dY[g][r][col0 + c] = 2 e / (B S)   (0 on padding rows / columns).
// grid = (blocks, members), one warp per row; partial[g][blockIdx.x] = the block's share of sum e^2 (fp64, fixed
// order), summed by train_sum_partials_kernel: the same inputs always give the same bits.
__global__ void __launch_bounds__(256)
train_loss_kernel(const float* __restrict__ pred, int DP, const float* __restrict__ state,
                  const float* __restrict__ next_state, int S, int B, int Bp, const float* __restrict__ d_mean,
                  const float* __restrict__ d_scale, float* __restrict__ dy, int OT, int col0, int width,
                  double* __restrict__ partial) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.y;
  const float gscale = 2.f / (static_cast<float>(B) * static_cast<float>(S));
  double acc = 0.0;
  for (int r = blockIdx.x * 8 + wib; r < Bp; r += gridDim.x * 8) {
    const long long row = static_cast<long long>(g) * Bp + r;
    float* drow = dy ? dy + row * OT + col0 : nullptr;
    for (int c = lane; c < width; c += 32) {
      float grad = 0.f;
      if (r < B && c < S) {
        const long long src = (static_cast<long long>(g) * B + r) * S + c;
        float t = next_state[src] - state[src];
        if (d_mean) t = (t - d_mean[c]) / d_scale[c];
        const float e = pred[row * DP + c] - t;
        acc += static_cast<double>(e) * e;
        grad = gscale * e;
      }
      if (drow) drow[c] = ptx::round_tf32(grad);
    }
  }
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  __shared__ double sh[8];
  if (lane == 0) sh[wib] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[w];
    partial[g * kTrainPartials + blockIdx.x] = t;
  }
}

// out[g] = scale * sum over regions r and slots b of partial[(r * n_members + g) * kTrainPartials + b]; one warp per
// member, fixed order.
__global__ void train_sum_partials_kernel(const double* __restrict__ partial, int regions, int n_members, double scale,
                                          double* __restrict__ out) {
  const int g = blockIdx.x, lane = threadIdx.x;
  if (g >= n_members || lane >= 32) return;
  double acc = 0.0;
  for (int r = 0; r < regions; ++r)
    for (int b = lane; b < kTrainPartials; b += 32) acc += partial[(static_cast<long long>(r) * n_members + g) * kTrainPartials + b];
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) out[g] = scale * acc;
}

// dst[z][c][r] = src[z][r][c] for r < rows, c < cols (32 x 32 tiles through shared memory); blockIdx.z = batch.
__global__ void train_transpose_kernel(const float* __restrict__ src, long long src_batch, int src_pitch, int rows,
                                       int cols, float* __restrict__ dst, long long dst_batch, int dst_pitch) {
  __shared__ float tile[32][33];
  const float* s = src + blockIdx.z * src_batch;
  float* d = dst + blockIdx.z * dst_batch;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? s[static_cast<long long>(r) * src_pitch + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) d[static_cast<long long>(c) * dst_pitch + r] = tile[threadIdx.x][i];
  }
}

// Several transposes in one launch (the weight slices every dgrad reads): blockIdx.z = descriptor * batch + member.
struct TransposeDesc {
  const float* src;
  long long src_batch;
  int src_pitch, rows, cols;
  float* dst;
  long long dst_batch;
  int dst_pitch;
};
__global__ void train_transpose_batch_kernel(const TransposeDesc* __restrict__ descs, int batch) {
  __shared__ float tile[32][33];
  const TransposeDesc d = descs[blockIdx.z / batch];
  const int member = blockIdx.z % batch;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  if (c0 >= d.cols || r0 >= d.rows) return;
  const float* s = d.src + member * d.src_batch;
  float* o = d.dst + member * d.dst_batch;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < d.rows && c < d.cols) ? s[static_cast<long long>(r) * d.src_pitch + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < d.cols && r < d.rows) o[static_cast<long long>(c) * d.dst_pitch + r] = tile[threadIdx.x][i];
  }
}

// dY_j = dH (.) act'(h_j): relu' = [h > 0], tanh' = 1 - h^2, written as a tf32 operand into the gradient concat.
__global__ void train_mask_kernel(const float* __restrict__ dh, int dh_pitch, const float* __restrict__ hbuf,
                                  int h_pitch, int h_col0, int width, long long n_rows, int tanh_act,
                                  float* __restrict__ dy, int OT, int dy_col0) {
  const long long total = n_rows * width;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % width);
    const long long row = idx / width;
    const float hv = hbuf[row * h_pitch + h_col0 + c];
    const float d = dh[row * dh_pitch + c];
    const float m = tanh_act ? (1.f - hv * hv) : (hv > 0.f ? 1.f : 0.f);
    dy[row * OT + dy_col0 + c] = ptx::round_tf32(d * m);
  }
}

// out[row] = sum_c x[row][c] for c < cols (bias gradients = row sums of dY^T); one warp per row.
__global__ void train_rowsum_kernel(const float* __restrict__ x, int pitch, int cols, long long n_rows,
                                    float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long row = warp; row < n_rows; row += n_warps) {
    float acc = 0.f;
    for (int c = lane; c < cols; c += 32) acc += x[row * pitch + c];
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) out[row] = acc;
  }
}

struct OptimArgs {
  int kind;          // 0: SGD with Nesterov momentum (torch.optim.SGD(nesterov=True)), 1: Adam
  float lr;
  float momentum;    // SGD momentum / Adam beta1
  float beta2;
  float eps;
  float grad_clip;   // 0: off; else clip_grad_norm_(max_norm) over one member's parameters
  float weight_decay;  // L2 term added to the gradient, g + wd * w (torch.optim's weight_decay, not decoupled); 0: off
};

// Step-dependent optimiser quantities live on the device so that a captured CUDA graph of the training step can
// be replayed: every step starts with train_tick_kernel.
struct OptimState {
  long long step;    // optimiser steps taken, including the current one
  float bc1, bc2;    // Adam bias corrections 1 - beta^step
  int first_step;    // SGD: the momentum buffer starts as the gradient itself
  int skip;          // the update is a no-op (a replayed value-baseline step past the end of its epoch)
};

// One optimiser step begins: the step counter and the quantities derived from it.  Called by one thread.
__device__ inline void optim_tick(OptimState* st, float beta1, float beta2) {
  const long long t = st->step + 1;
  st->step = t;
  st->first_step = t == 1;
  st->bc1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), static_cast<double>(t)));
  st->bc2 = static_cast<float>(1.0 - pow(static_cast<double>(beta2), static_cast<double>(t)));
}

__global__ void train_tick_kernel(OptimState* st, float beta1, float beta2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) optim_tick(st, beta1, beta2);
}

// Every parameter tensor of the ensemble in one launch: blockIdx.z = tensor, blockIdx.y = member.  Member g's
// parameters sit at p[g * p_stride + i], its gradient and optimiser moments at {g, m, v}[g * g_stride + g_off + i].
// The norm kernel writes fixed-order block partials (gradient norm, dynamics.py:247-248); the update applies
//   coef = min(1, clip / (sqrt(sumsq) + 1e-6))    (torch.nn.utils.clip_grad_norm_)
// and then SGD-Nesterov or Adam.
struct ParamDesc {
  float* p;         // parameters, member stride p_stride
  const float* g;   // gradient; {g, m, v}[member * g_stride + g_off + i]
  float* m;
  float* v;
  long long count, p_stride, g_stride, g_off;
};

__global__ void __launch_bounds__(256)
train_sumsq_batch_kernel(const ParamDesc* __restrict__ descs, int n_members, double* __restrict__ partial) {
  const ParamDesc d = descs[blockIdx.z];
  const int g = blockIdx.y;
  const float* p = d.g + g * d.g_stride + d.g_off;
  double acc = 0.0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < d.count;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const double v = p[i];
    acc += v * v;
  }
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  __shared__ double sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[w];
    partial[(static_cast<long long>(blockIdx.z) * n_members + g) * kTrainPartials + blockIdx.x] = t;
  }
}

__global__ void train_optim_batch_kernel(const ParamDesc* __restrict__ descs, int n_members,
                                         const double* __restrict__ sumsq, const OptimArgs a,
                                         const OptimState* __restrict__ state) {
  const ParamDesc d = descs[blockIdx.z];
  const int gi = blockIdx.y;
  const OptimState os = *state;
  if (os.skip) return;
  float coef = 1.f;
  if (a.grad_clip > 0.f) {
    const float c = a.grad_clip / (static_cast<float>(sqrt(sumsq[gi])) + 1e-6f);
    coef = c < 1.f ? c : 1.f;
  }
  float* pp = d.p + gi * d.p_stride;
  const long long gbase = gi * d.g_stride + d.g_off;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < d.count;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float grad = d.g[gbase + i] * coef;
    float w = pp[i];
    if (a.weight_decay != 0.f) grad = fmaf(a.weight_decay, w, grad);
    if (a.kind == 0) {
      const float buf = os.first_step ? grad : fmaf(a.momentum, d.m[gbase + i], grad);
      d.m[gbase + i] = buf;
      w -= a.lr * fmaf(a.momentum, buf, grad);
    } else {
      const float m1 = fmaf(a.momentum, d.m[gbase + i], (1.f - a.momentum) * grad);
      const float v1 = fmaf(a.beta2, d.v[gbase + i], (1.f - a.beta2) * grad * grad);
      d.m[gbase + i] = m1;
      d.v[gbase + i] = v1;
      const float denom = sqrtf(v1) / sqrtf(os.bc2) + a.eps;
      w -= (a.lr / os.bc1) * (m1 / denom);
    }
    pp[i] = w;
  }
}

// Packed operand rows -> nn.Linear layout (inverse of pack_weight_kernel): dst[o][src0 + i] = src[o][dst0 + i].
__global__ void train_unpack_kernel(const float* __restrict__ packed, long long packed_pitch, int rows,
                                    float* __restrict__ out, int out_pitch, PackSegs segs) {
  const int o = blockIdx.x;
  if (o >= rows) return;
  for (int s = 0; s < segs.n; ++s)
    for (int i = threadIdx.x; i < segs.width[s]; i += blockDim.x)
      out[static_cast<long long>(o) * out_pitch + segs.src0[s] + i] = packed[o * packed_pitch + segs.dst0[s] + i];
}

}  // namespace simstep
