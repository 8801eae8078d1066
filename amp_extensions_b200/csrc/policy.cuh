// Gaussian MLP policy of the rollout loop (reference mjrl/mjrl/policies/gaussian_mlp.py:95-104 over
// mjrl/mjrl/utils/fc_network.py:42-55):
//     x = (obs - in_shift) / (in_scale + 1e-8);  h = act(W_l h + b_l) for the hidden layers;
//     mean = (W_L h + b_L) * out_scale + out_shift;  action = mean + exp(log_std) * noise.
// The network is tiny (226 -> 32 -> 32 -> 28 in MILO's runs: 9 k multiply-adds per env), so it runs in plain fp32
// on the CUDA cores with the reference's own rounding of every layer: weights sit transposed in shared
// memory, a warp evaluates four envs at a time with lanes = output units, activations of the four envs are
// broadcast from shared memory as one float4.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ptx.cuh"

namespace simstep {

constexpr int kPolicyMaxLayers = 4;   // linear layers (hidden + output)
constexpr int kPolicyMaxWidth = 128;  // widest hidden / output layer
constexpr int kPolicyMaxIn = 512;     // observation width
constexpr int kPolicyWarps = 4;
constexpr int kPolicyEnvsPerWarp = 4;

struct PolicyConst {
  int n_layers;                       // linear layers
  int in_dim[kPolicyMaxLayers];
  int out_dim[kPolicyMaxLayers];
  int out_pad[kPolicyMaxLayers];      // out_dim rounded up to 32: row stride of the transposed weights
  int w_off[kPolicyMaxLayers];        // float offset of layer l's transposed weights [in][out_pad] in the pack
  int b_off[kPolicyMaxLayers];        // float offset of layer l's bias [out_pad]
  int pack_floats;                    // total floats of the parameter pack
  int tanh_act;                       // 1 tanh, 0 relu (fc_network.py:30)
  int obs_dim, act_dim;
};

inline size_t policy_smem_bytes(const PolicyConst& c) {
  // parameter pack + per warp two activation buffers of [max width][4 envs]
  const int width = c.obs_dim > kPolicyMaxWidth ? c.obs_dim : kPolicyMaxWidth;
  return (size_t(c.pack_floats) + size_t(kPolicyWarps) * 2 * width * kPolicyEnvsPerWarp) * sizeof(float);
}

// pack:   per layer transposed weights and bias as laid out by PolicyConst, then
//         in_shift [obs_dim] | in_div [obs_dim] (= in_scale + 1e-8) | out_scale [act] | out_shift [act] | std [act]
__global__ void __launch_bounds__(kPolicyWarps * 32)
policy_act_kernel(const PolicyConst c, const float* __restrict__ pack, const float* __restrict__ tail,
                  const float* __restrict__ obs, const float* __restrict__ noise, long long n_envs,
                  float* __restrict__ action, float* __restrict__ mean_out) {
  extern __shared__ __align__(16) float sm_pol[];
  float* s_pack = sm_pol;
  const int width = c.obs_dim > kPolicyMaxWidth ? c.obs_dim : kPolicyMaxWidth;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* buf0 = sm_pol + c.pack_floats + size_t(warp) * 2 * width * kPolicyEnvsPerWarp;
  float* buf1 = buf0 + width * kPolicyEnvsPerWarp;
  for (int i = threadIdx.x; i < c.pack_floats; i += blockDim.x) s_pack[i] = pack[i];  // parameters: not produced by
  ptx::grid_dep_wait();                                                               // the previous kernel
  ptx::grid_dep_launch();
  __syncthreads();
  const float* in_shift = tail;
  const float* in_div = tail + c.obs_dim;
  const float* out_scale = in_div + c.obs_dim;
  const float* out_shift = out_scale + c.act_dim;
  const float* stdv = out_shift + c.act_dim;

  const long long n_groups = (n_envs + kPolicyEnvsPerWarp - 1) / kPolicyEnvsPerWarp;
  for (long long grp = blockIdx.x * static_cast<long long>(kPolicyWarps) + warp; grp < n_groups;
       grp += static_cast<long long>(gridDim.x) * kPolicyWarps) {
    const long long e0 = grp * kPolicyEnvsPerWarp;
    __syncwarp();
    // normalised observations of the group's envs -> buf0[k][r]
    for (int r = 0; r < kPolicyEnvsPerWarp; ++r) {
      const long long e = e0 + r;
      for (int k = lane; k < c.obs_dim; k += 32) {
        const float v = e < n_envs ? (obs[e * c.obs_dim + k] - in_shift[k]) / in_div[k] : 0.f;
        buf0[k * kPolicyEnvsPerWarp + r] = v;
      }
    }
    __syncwarp();
    float* cur = buf0;
    float* nxt = buf1;
    for (int l = 0; l < c.n_layers; ++l) {
      const float* W = s_pack + c.w_off[l];
      const float* B = s_pack + c.b_off[l];
      const int K = c.in_dim[l], O = c.out_dim[l], OP = c.out_pad[l];
      const bool last = l == c.n_layers - 1;
      for (int o = lane; o < OP; o += 32) {
        float a0 = B[o], a1 = a0, a2 = a0, a3 = a0;
        // nn.Linear accumulates the dot product then adds the bias; fp32 summation order differs from
        // ATen's sgemm only by rounding (<< 1e-6 relative at these widths)
        float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll 4
        for (int k = 0; k < K; ++k) {
          const float w = W[k * OP + o];
          const float4 x = *reinterpret_cast<const float4*>(cur + k * kPolicyEnvsPerWarp);
          d0 = fmaf(w, x.x, d0); d1 = fmaf(w, x.y, d1); d2 = fmaf(w, x.z, d2); d3 = fmaf(w, x.w, d3);
        }
        a0 += d0; a1 += d1; a2 += d2; a3 += d3;
        if (o < O) {
          if (!last) {
            if (c.tanh_act) { a0 = tanhf(a0); a1 = tanhf(a1); a2 = tanhf(a2); a3 = tanhf(a3); }
            else { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); a2 = fmaxf(a2, 0.f); a3 = fmaxf(a3, 0.f); }
            *reinterpret_cast<float4*>(nxt + o * kPolicyEnvsPerWarp) = make_float4(a0, a1, a2, a3);
          } else {
            const float sc = out_scale[o], sh = out_shift[o], sd = stdv[o];
            const float m[4] = {fmaf(a0, sc, sh), fmaf(a1, sc, sh), fmaf(a2, sc, sh), fmaf(a3, sc, sh)};
#pragma unroll
            for (int r = 0; r < kPolicyEnvsPerWarp; ++r) {
              const long long e = e0 + r;
              if (e < n_envs) {
                if (mean_out) mean_out[e * c.act_dim + o] = m[r];
                if (action) action[e * c.act_dim + o] = noise ? fmaf(sd, noise[e * c.act_dim + o], m[r]) : m[r];
              }
            }
          }
        }
      }
      __syncwarp();
      float* t = cur; cur = nxt; nxt = t;
    }
  }
}

// Reverse discounted sums over time-major [T][E] arrays, one thread per env (reference
// mjrl/mjrl/utils/process_samples.py:3-45).  An env's column holds one or more trajectories back to back:
// seg_end[t][e] != 0 marks the last step of a trajectory that TERMINATED (sampler.py:79 stores terminated=done);
// the trailing trajectory ends at len[e]-1 and counts as terminated iff terminated[e] != 0.  Per trajectory
//     returns[t]    = reward[t] + gamma * returns[t+1]                                  (discount_sum)
//     advantages[t] = delta[t] + gamma*lambda * advantages[t+1],
//     delta[t]      = reward[t] + gamma * b1[t+1] - baseline[t],  b1[end+1] = terminated ? 0 : baseline[end]
// entries at t >= len[e] are written as 0.
__global__ void discount_kernel(const float* __restrict__ reward, const float* __restrict__ baseline,
                                const uint8_t* __restrict__ seg_end, const int32_t* __restrict__ len,
                                const uint8_t* __restrict__ terminated, int T, long long n_envs, float gamma,
                                float gae_lambda, float* __restrict__ returns, float* __restrict__ advantages) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < n_envs;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int L = len ? min(max(len[e], 0), T) : T;
    float ret = 0.f, adv = 0.f;
    float b_next = 0.f;
    if (baseline && L > 0 && !(terminated && terminated[e])) b_next = baseline[static_cast<long long>(L - 1) * n_envs + e];
    for (int t = T - 1; t >= 0; --t) {
      const long long i = static_cast<long long>(t) * n_envs + e;
      if (t >= L) {
        if (returns) returns[i] = 0.f;
        if (advantages) advantages[i] = 0.f;
        continue;
      }
      if (seg_end && seg_end[i]) { ret = 0.f; adv = 0.f; b_next = 0.f; }  // a terminated trajectory ends here
      const float r = reward[i];
      ret = fmaf(gamma, ret, r);
      if (returns) returns[i] = ret;
      if (advantages) {
        const float b = baseline[i];
        const float delta = r + gamma * b_next - b;
        adv = fmaf(gamma * gae_lambda, adv, delta);
        advantages[i] = adv;
        b_next = b;
      }
    }
  }
}

// Auto-reset between two steps of the rollout loop (reference milo/milo/sampler.py:36-66 starts a new trajectory
// with env.reset(), gym-simenv/gym_simenv/envs/sim_env.py:270-285: fresh initial state, num_steps = 0, member
// round-robin).  One warp per env row:
//     done[e] ? (state_out[e] = pool[pick[e] % n_pool], num_steps[e] = 0, member[e] = (member[e]+1) % n_models)
//             : (state_out[e] = next_state[e])
__global__ void __launch_bounds__(256)
auto_reset_kernel(const float* __restrict__ next_state, const uint8_t* __restrict__ done,
                  const float* __restrict__ pool, const int32_t* __restrict__ pick, int n_pool, int n_models, int S,
                  long long n_envs, float* __restrict__ state_out, int32_t* __restrict__ member,
                  int32_t* __restrict__ num_steps) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const int lane = threadIdx.x & 31;
  const long long warp0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5;
  const long long n_warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const bool vec2 = (S % 2 == 0) && (reinterpret_cast<uintptr_t>(next_state) % 8 == 0) &&
                    (reinterpret_cast<uintptr_t>(pool) % 8 == 0) && (reinterpret_cast<uintptr_t>(state_out) % 8 == 0);
  for (long long e = warp0; e < n_envs; e += n_warps) {
    const bool d = done[e] != 0;
    const float* src = next_state + e * S;
    if (d) {
      int p = pick[e] % n_pool;
      if (p < 0) p += n_pool;
      src = pool + static_cast<long long>(p) * S;
      if (lane == 0) {
        if (num_steps) num_steps[e] = 0;
        if (member) member[e] = (member[e] + 1) % n_models;
      }
    }
    float* dst = state_out + e * S;
    if (vec2) {
      const float2* s2 = reinterpret_cast<const float2*>(src);
      float2* d2 = reinterpret_cast<float2*>(dst);
      for (int k = lane; k < S / 2; k += 32) d2[k] = s2[k];
    } else {
      for (int k = lane; k < S; k += 32) dst[k] = src[k];
    }
  }
}

// Moments of a (masked) vector for advantage whitening (mjrl/mjrl/utils/process_samples.py:14-19, 31-36:
// alladv.mean(), alladv.std()) and rollout statistics: two deterministic passes, fp64 accumulation.
//   pass 1: partial[b] = {count, sum, sum of squares} of block b's grid-stride slice
//   pass 2: out[0..2] = sum over blocks (fixed order)
constexpr int kMomentsThreads = 256;
constexpr int kMomentsMaxBlocks = 1024;

__global__ void __launch_bounds__(kMomentsThreads)
moments_partial_kernel(const float* __restrict__ x, const uint8_t* __restrict__ valid, long long n,
                       double* __restrict__ partial) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  double c = 0.0, s = 0.0, q = 0.0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (valid == nullptr || valid[i]) {
      const double v = x[i];
      c += 1.0;
      s += v;
      q += v * v;
    }
  }
  __shared__ double sh[3][kMomentsThreads / 32];
  for (int off = 16; off > 0; off >>= 1) {
    c += __shfl_xor_sync(0xffffffffu, c, off);
    s += __shfl_xor_sync(0xffffffffu, s, off);
    q += __shfl_xor_sync(0xffffffffu, q, off);
  }
  if ((threadIdx.x & 31) == 0) {
    sh[0][threadIdx.x >> 5] = c;
    sh[1][threadIdx.x >> 5] = s;
    sh[2][threadIdx.x >> 5] = q;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int w = 0; w < kMomentsThreads / 32; ++w) t += sh[threadIdx.x][w];
    partial[blockIdx.x * 3 + threadIdx.x] = t;
  }
}

__global__ void moments_final_kernel(const double* __restrict__ partial, int n_blocks, double* __restrict__ out) {
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int b = 0; b < n_blocks; ++b) t += partial[b * 3 + threadIdx.x];
    out[threadIdx.x] = t;
  }
}

// out = (x - mean) / (std + eps) with mean / population std from stats = {count, sum, sum of squares} (fp64, e.g.
// the all-reduced output of moments); masked-out entries are written as 0.
__global__ void whiten_kernel(const float* __restrict__ x, const uint8_t* __restrict__ valid, long long n,
                              const double* __restrict__ stats, float eps, float* __restrict__ out) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  const double cnt = stats[0] > 0.0 ? stats[0] : 1.0;
  const double mean = stats[1] / cnt;
  const double var = stats[2] / cnt - mean * mean;
  const double sd = sqrt(var > 0.0 ? var : 0.0);
  const float m = static_cast<float>(mean);
  const float inv = static_cast<float>(1.0 / (sd + static_cast<double>(eps)));
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    out[i] = (valid == nullptr || valid[i]) ? (x[i] - m) * inv : 0.f;
}

// Fixed-range histogram (simstep_histogram): counts[b] += #{i : x[i] in [lo, hi],
// bin(x[i]) == b}, bin = clamp(floor((x - lo) / width), 0, bins - 1) evaluated in fp64.  Integer
// counts: the result does not depend on scheduling.  Shared-memory bins per block, then one atomic per non-empty bin.
constexpr int kHistMaxBins = 8192;

__global__ void __launch_bounds__(256)
histogram_kernel(const float* __restrict__ x, long long n, double lo, double hi, int bins,
                 unsigned long long* __restrict__ counts) {
  extern __shared__ unsigned int sh_bins[];
  for (int b = threadIdx.x; b < bins; b += blockDim.x) sh_bins[b] = 0u;
  __syncthreads();
  const double width = (hi - lo) / bins;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const double v = x[i];
    if (v >= lo && v <= hi) {
      int b = static_cast<int>(floor((v - lo) / width));
      b = b < 0 ? 0 : (b >= bins ? bins - 1 : b);
      atomicAdd(&sh_bins[b], 1u);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < bins; b += blockDim.x)
    if (sh_bins[b]) atomicAdd(&counts[b], static_cast<unsigned long long>(sh_bins[b]));
}


// ---- device-side steps of the distributed quantile (parallel.global_quantile) --------------------------------
// Exact radix selection on the order-preserving key of the fp32 bit pattern,
//     key(u) = u ^ (sign(u) ? 0xFFFFFFFF : 0x80000000)      (unsigned order of keys = order of the floats),
// NaN (detected on the bits before keying) counted in a slot of its own.  Three histogram passes of 12, 12 and 8
// key bits fix all 32 bits of the two order statistics that bracket the quantile.
// qstate (doubles, resident on the device): [0] q (set by the caller), [1] result (written by the SELECT that fixes
// the last bits), [2] n, [3] NaN count; order statistic i in {0, 1}: [4 + 4i] key prefix, [5 + 4i] key bits fixed
// (32 = done), [6 + 4i] samples whose key is below the prefix, [7 + 4i] rank k.  Start: q, then zeros.
constexpr int kQuantileBins = 4096;                      // widest digit: 12 bits
constexpr int kQuantileNanSlot = 2 * kQuantileBins;      // counts: [2][kQuantileBins] + NaN count
constexpr int kQuantileDigit = 12;

__device__ __forceinline__ int quantile_digit_bits(int fixed) { return min(kQuantileDigit, 32 - fixed); }

// counts[i * kQuantileBins + d] += samples whose key matches prefix i and has next digit d; while both order
// statistics share their prefix (always in the first pass) only window 0 is counted.  The first pass also counts NaN.
// Equal digits of a warp are combined with __match_any_sync before the shared-memory atomic (heavy ties, e.g.
// exact zeros, would otherwise serialise a warp on one bin).
__global__ void __launch_bounds__(256)
quantile_hist_kernel(const float* __restrict__ x, long long n, const double* __restrict__ qstate,
                     unsigned long long* __restrict__ counts) {
  __shared__ unsigned int sh_bins[2 * kQuantileBins + 1];
  int fixed[2];
  unsigned prefix[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    prefix[i] = static_cast<unsigned>(qstate[4 + 4 * i]);
    fixed[i] = static_cast<int>(qstate[5 + 4 * i]);
  }
  if (fixed[0] >= 32 && fixed[1] >= 32) return;
  const int windows = (fixed[0] == fixed[1] && prefix[0] == prefix[1]) ? 1 : 2;
  const bool count_nan = fixed[0] == 0;
  for (int b = threadIdx.x; b < 2 * kQuantileBins + 1; b += blockDim.x) sh_bins[b] = 0u;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  // every thread of a block runs the same number of iterations: the warp votes below need all lanes
  for (long long base = blockIdx.x * static_cast<long long>(blockDim.x); base < n;
       base += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long j = base + threadIdx.x;
    const bool valid = j < n;
    const unsigned u = valid ? __float_as_uint(x[j]) : 0u;
    const bool nan = valid && (u & 0x7fffffffu) > 0x7f800000u;
    const unsigned key = u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
    if (count_nan) {
      const unsigned m = __ballot_sync(0xffffffffu, nan);
      if (lane == 0 && m) atomicAdd(&sh_bins[kQuantileNanSlot], static_cast<unsigned>(__popc(m)));
    }
    for (int i = 0; i < windows; ++i) {
      int bin = -1;
      if (valid && !nan && fixed[i] < 32 && (fixed[i] == 0 || (key >> (32 - fixed[i])) == prefix[i])) {
        const int w = quantile_digit_bits(fixed[i]);
        bin = static_cast<int>((key >> (32 - fixed[i] - w)) & ((1u << w) - 1u));
      }
      const unsigned peers = __match_any_sync(0xffffffffu, bin);
      if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(&sh_bins[i * kQuantileBins + bin], static_cast<unsigned>(__popc(peers)));
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < 2 * kQuantileBins + 1; b += blockDim.x)
    if (sh_bins[b]) atomicAdd(&counts[b], static_cast<unsigned long long>(sh_bins[b]));
}

__device__ __forceinline__ double quantile_key_value(unsigned key) {
  return static_cast<double>(__uint_as_float((key & 0x80000000u) ? (key ^ 0x80000000u) : ~key));
}

// Given the (all-reduced) counts of one HIST pass: in the first pass n, the NaN count and the ranks
// k0 = floor(q (n - 1)), k1 = min(k0 + 1, n - 1); then appends to each prefix the digit whose cumulative count
// (plus the samples below the prefix) first exceeds k.  When the last bits are fixed, qstate[1] = the
// quantile, interpolated in fp64 with torch.lerp's formula; NaN when there are no samples or any NaN.
// One block; thread t sums a contiguous run of bins, thread 0 walks the runs, then the bins of the run.
__global__ void __launch_bounds__(256)
quantile_select_kernel(const long long* __restrict__ counts, double* __restrict__ qstate) {
  __shared__ long long run_sum[256];
  const bool same = qstate[4] == qstate[8] && qstate[5] == qstate[9];
  bool finished = false;
  for (int i = 0; i < 2; ++i) {
    double* st = qstate + 4 + 4 * i;
    const int fixed = static_cast<int>(st[1]);  // the same in every thread: written by thread 0 before a barrier
    if (fixed >= 32) continue;
    const int w = quantile_digit_bits(fixed);
    const int nb = 1 << w;
    const int per = nb / 256;
    const long long* c = counts + (same ? 0 : i * kQuantileBins);
    long long s = 0;
    for (int b = threadIdx.x * per; b < (threadIdx.x + 1) * per; ++b) s += c[b];
    run_sum[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      bool active = true;
      if (fixed == 0 && i == 0) {
        long long valid = 0;
        for (int t = 0; t < 256; ++t) valid += run_sum[t];
        const long long nan = counts[kQuantileNanSlot];
        const long long n = valid + nan;
        qstate[2] = static_cast<double>(n);
        qstate[3] = static_cast<double>(nan);
        if (nan > 0 || n == 0) {
          qstate[1] = NAN;
          qstate[5] = qstate[9] = 32.0;
          active = false;
        } else {
          const double k0 = floor(qstate[0] * static_cast<double>(n - 1));
          qstate[7] = k0;
          qstate[11] = fmin(k0 + 1.0, static_cast<double>(n - 1));
        }
      }
      if (active) {
        const long long k = static_cast<long long>(st[3]);
        long long cum = static_cast<long long>(st[2]);
        int t = 0;
        while (t < 255 && cum + run_sum[t] <= k) cum += run_sum[t++];
        int b = t * per;
        while (b < (t + 1) * per - 1 && cum + c[b] <= k) cum += c[b++];
        st[0] = st[0] * nb + b;
        st[1] = fixed + w;
        st[2] = static_cast<double>(cum);
        finished = fixed + w == 32;
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0 && finished) {  // both order statistics advance together: window 1 fixed its last bits
    const double v0 = quantile_key_value(static_cast<unsigned>(qstate[4]));
    const double v1 = quantile_key_value(static_cast<unsigned>(qstate[8]));
    const double pos = qstate[0] * (qstate[2] - 1.0);
    const double wt = pos - floor(pos);
    const double d = v1 - v0;
    // torch.lerp: self + w (end - self) for w < 0.5, else end - (end - self)(1 - w); w == 0 is sorted[k0] exactly
    qstate[1] = wt == 0.0 ? v0 : (wt < 0.5 ? fma(wt, d, v0) : fma(-d, 1.0 - wt, v1));
  }
}

}  // namespace simstep
