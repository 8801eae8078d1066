// Natural policy gradient step of mjrl's Gaussian MLP policy on the device (mjrl/mjrl/algos/npg_cg.py: NPG.train_from_paths,
// NPG.HVP / build_Hvp_eval, NPG.flat_vpg, NPG.CPI_surrogate, NPG.kl_old_new; mjrl/mjrl/utils/cg_solve.py: cg_solve;
// mjrl/mjrl/policies/gaussian_mlp.py: MLP.log_likelihood, MLP.mean_kl, MLP.set_param_values).
//
// The policy is the one of policy.cuh (transposed pack [in][out_pad] + bias per layer, tail in_shift | in_div |
// out_scale | out_shift | std).  Every row kernel processes tiles of R rows (R = 32 or 64) with one CTA of 512 threads:
//   * activations of a tile live in shared memory row-major [r][feature], feature stride = 4 mod 8 floats (float4 rows,
//     conflict-free per-lane float4 loads); every layer input carries a constant-1 column at feature in_l, so the bias
//     is row in_l of the transposed pack and the bias gradient is column in_l of the weight gradient;
//   * forward / JVP / backward-data products run with lane = row and a warp per (row half, 4 output units), the
//     weights broadcast from shared memory as float4 (the same fp32 FMA scheme as policy_act_kernel);
//   * weight gradients G_l[o][k] += sum_r delta_l[r][o] a_l[r][k] are 4x4 blocks owned by fixed threads for the whole
//     kernel, accumulated in registers over every tile the CTA sees, written once to partial[block][...] at the end.
// No atomics anywhere: the per-CTA partials are summed in a fixed order in fp64 by npg_reduce_kernel, so a result is
// bit-identical from run to run.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "policy.cuh"
#include "ptx.cuh"

namespace simstep {

constexpr int kNpgThreads = 512;
constexpr int kNpgWarps = kNpgThreads / 32;
constexpr int kNpgMaxItems = 3;                       // 4x4 gradient blocks per thread (48 accumulator registers)
constexpr int kNpgMaxBlocks = kNpgThreads * kNpgMaxItems;
constexpr int kNpgMaxRows = 64;                       // rows per tile: 64, or 32 when that plan does not fit
constexpr int kNpgExtra = 4;                          // per-row scalar sums after the log_std entries
constexpr int kNpgCgThreads = 1024;

enum NpgMode { kNpgGrad = 0, kNpgPrep = 1, kNpgFvp = 2, kNpgDiag = 3 };

// [r][feature] stride of a tile with `w` columns: float4 aligned, = 4 mod 8 (8 lanes of a float4 phase hit distinct banks)
__host__ __device__ inline int npg_stride(int w) { return (w + 7) / 8 * 8 + 4; }

struct NpgConst {
  PolicyConst c;
  int R;                                  // rows per tile (32 or 64)
  int a_off[kPolicyMaxLayers];            // smem float offset of layer l's input tile a_l [R][sa_l]
  int sa[kPolicyMaxLayers];
  int da_off[kPolicyMaxLayers];           // FVP: tangent of a_l (l >= 1)
  int d_off[kPolicyMaxLayers];            // delta_l [R][sd_l], cotangent of layer l's pre-activation
  int sd[kPolicyMaxLayers];
  int e_off, se;                          // per-row scalars [R][se]: log_std terms (A) then kNpgExtra sums
  int pack_pad;                           // floats of the pack copy in shared memory (multiple of 4)
  int smem_floats;
  int blk0[kPolicyMaxLayers + 1];         // first 4x4 gradient block of layer l; blk0[n_layers] = total blocks
  int kq[kPolicyMaxLayers];               // k-quads of layer l: ceil((in_l + 1) / 4)
  int cache_off[kPolicyMaxLayers];        // float offset of hidden activation a_l (l >= 1) in a cache row
  int cache_w;                            // floats per cache row (sum of hidden widths)
  int pstride;                            // floats per CTA partial: 16 * blocks + act_dim + kNpgExtra, rounded to 4
};

struct NpgArgs {
  const float* obs;        // [n][obs_dim]
  const float* act;        // [n][act_dim]   (GRAD, DIAG)
  const float* adv;        // [n]            (GRAD, DIAG)
  const uint8_t* valid;    // [n] or null
  long long n;
  const int64_t* idx;      // Fisher rows (PREP, FVP): null = rows 0..n-1
  long long n_rows;        // rows the kernel walks: n, or the number of Fisher indices
  float* cache;            // [n_rows][cache_w] hidden activations of the Fisher rows (PREP writes, FVP reads)
  const float* vpack;      // FVP: direction in pack layout
  const float* old_pack;   // DIAG: parameters before the step (pack layout, global)
  const float* old_tail;   // DIAG: std before the step [act]
  const float* ls_new;     // DIAG: log_std after / before the step [act]
  const float* ls_old;
  const int* skip;         // FVP in CG mode: nonzero -> CG has converged, the launch does nothing
  float* partial;          // [gridDim.x][pstride]
};

// acc[0..3] += sum_{k < K} x[k] * Wt[k][o0 .. o0 + 3]   (x: this lane's row, Wt row stride OP)
__device__ __forceinline__ void npg_mac_rows(float acc[4], const float* __restrict__ x, int K,
                                             const float* __restrict__ Wt, int OP, int o0) {
  int k = 0;
#pragma unroll 1
  for (; k + 4 <= K; k += 4) {
    const float4 xv = *reinterpret_cast<const float4*>(x + k);
    const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 w = *reinterpret_cast<const float4*>(Wt + (k + i) * OP + o0);
      acc[0] = fmaf(xs[i], w.x, acc[0]);
      acc[1] = fmaf(xs[i], w.y, acc[1]);
      acc[2] = fmaf(xs[i], w.z, acc[2]);
      acc[3] = fmaf(xs[i], w.w, acc[3]);
    }
  }
  for (; k < K; ++k) {
    const float4 w = *reinterpret_cast<const float4*>(Wt + k * OP + o0);
    const float xs = x[k];
    acc[0] = fmaf(xs, w.x, acc[0]);
    acc[1] = fmaf(xs, w.y, acc[1]);
    acc[2] = fmaf(xs, w.z, acc[2]);
    acc[3] = fmaf(xs, w.w, acc[3]);
  }
}

// acc[i] += sum_{o < O4} d[o] * Wt[k0 + i][o]   (backward data product W^T delta for inputs k0 .. k0 + 3)
__device__ __forceinline__ void npg_mac_back(float acc[4], const float* __restrict__ d, int O4,
                                             const float* __restrict__ Wt, int OP, int k0, int kmax) {
#pragma unroll 1
  for (int o = 0; o < O4; o += 4) {
    const float4 dv = *reinterpret_cast<const float4*>(d + o);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (k0 + i < kmax) {
        const float4 w = *reinterpret_cast<const float4*>(Wt + (k0 + i) * OP + o);
        acc[i] = fmaf(dv.x, w.x, fmaf(dv.y, w.y, fmaf(dv.z, w.z, fmaf(dv.w, w.w, acc[i]))));
      }
    }
  }
}

__device__ __forceinline__ float npg_act_grad(int tanh_act, float h) { return tanh_act ? 1.f - h * h : (h > 0.f ? 1.f : 0.f); }

template <int MODE>
__global__ void __launch_bounds__(kNpgThreads, 1)
npg_rows_kernel(const NpgConst q, const float* __restrict__ pack, const float* __restrict__ tail, const NpgArgs a) {
  extern __shared__ __align__(16) float sm_npg[];
  const PolicyConst& c = q.c;
  const int L = c.n_layers, A = c.act_dim, R = q.R;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Wt = sm_npg;
  ptx::grid_dep_wait();  // the parameters may have been written by the previous kernel (apply / set)
  ptx::grid_dep_launch();
  if (MODE == kNpgFvp && a.skip && *a.skip) return;
  for (int i = threadIdx.x; i < c.pack_floats; i += blockDim.x) Wt[i] = pack[i];
  for (int i = q.pack_pad + threadIdx.x; i < q.smem_floats; i += blockDim.x) sm_npg[i] = 0.f;  // pads stay 0
  const float* in_shift = tail;
  const float* in_div = tail + c.obs_dim;
  const float* out_scale = in_div + c.obs_dim;
  const float* out_shift = out_scale + c.act_dim;
  const float* stdv = out_shift + c.act_dim;
  float* E = sm_npg + q.e_off;

  float acc[kNpgMaxItems][16];
#pragma unroll
  for (int j = 0; j < kNpgMaxItems; ++j)
#pragma unroll
    for (int e = 0; e < 16; ++e) acc[j][e] = 0.f;
  float ext = 0.f;  // thread t < A + kNpgExtra owns per-row scalar column t
  // source row of each tile row: idx[row] or row; -1 past n_rows or masked out by `valid`.  A masked row enters the
  // tile as zeros, like a row past the end, so whatever it holds (NaN, Inf) never reaches a product that is summed.
  __shared__ long long s_src[kNpgMaxRows];

  const long long n_tiles = (a.n_rows + R - 1) / R;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long r0 = tile * R;
    for (int r = threadIdx.x; r < R; r += blockDim.x) {  // last read by the previous tile's output stage, then a barrier
      const long long row = r0 + r;
      long long src = -1;
      if (row < a.n_rows) {
        src = a.idx ? a.idx[row] : row;
        if (a.valid && !a.valid[src]) src = -1;
      }
      s_src[r] = src;
    }
    __syncthreads();  // the previous tile's tiles are consumed
    // ---- input rows: normalised observations, the constant-1 column, and (FVP) the cached hidden activations
    {
      float* a0 = sm_npg + q.a_off[0];
      const int sa0 = q.sa[0];
      for (int i = threadIdx.x; i < R * c.obs_dim; i += blockDim.x) {
        const int r = i / c.obs_dim, k = i - r * c.obs_dim;
        const long long src = s_src[r];
        a0[r * sa0 + k] = src >= 0 ? (a.obs[src * c.obs_dim + k] - in_shift[k]) / in_div[k] : 0.f;
      }
      for (int l = 0; l < L; ++l)
        for (int r = threadIdx.x; r < R; r += blockDim.x) {
          sm_npg[q.a_off[l] + r * q.sa[l] + c.in_dim[l]] = 1.f;
          if (MODE == kNpgDiag && l > 0) sm_npg[q.da_off[l] + r * q.sa[l] + c.in_dim[l]] = 1.f;
        }
      if (MODE == kNpgFvp) {
        for (int l = 1; l < L; ++l) {
          const int w = c.in_dim[l];
          for (int i = threadIdx.x; i < R * w; i += blockDim.x) {
            const int r = i / w, k = i - r * w;
            const long long row = r0 + r;
            sm_npg[q.a_off[l] + r * q.sa[l] + k] = s_src[r] >= 0 ? a.cache[row * q.cache_w + q.cache_off[l] + k] : 0.f;
          }
        }
      }
    }
    __syncthreads();
    // ---- forward (GRAD / PREP / DIAG) or tangent (FVP) layer by layer; the last layer's result goes to delta_{L-1}
    for (int l = 0; l < L; ++l) {
      const int K = c.in_dim[l], O = c.out_dim[l], OP = c.out_pad[l];
      const bool last = l == L - 1;
      const int nq = (O + 3) / 4;
      const int units = (R / 32) * nq;
      const float* Wl = Wt + c.w_off[l];
      const int sa = q.sa[l];
      for (int u = warp; u < units; u += kNpgWarps) {
        const int half = u / nq, o0 = (u - half * nq) * 4;
        const int r = half * 32 + lane;
        const float* x = sm_npg + q.a_off[l] + r * sa;
        float y[4] = {0.f, 0.f, 0.f, 0.f};
        if (MODE == kNpgFvp) {
          npg_mac_rows(y, x, K + 1, a.vpack + c.w_off[l], OP, o0);      // V_l a_l + vb_l
          if (l > 0) npg_mac_rows(y, sm_npg + q.da_off[l] + r * sa, K, Wl, OP, o0);  // + W_l da_l
        } else {
          npg_mac_rows(y, x, K + 1, Wl, OP, o0);                        // W_l a_l + b_l
        }
        if constexpr (MODE == kNpgDiag) {  // the old parameters' pre-activation goes beside the new one
          float yo[4] = {0.f, 0.f, 0.f, 0.f};
          const float* xo = sm_npg + q.da_off[l] + r * sa;  // da_l doubles as the old forward's activations
          npg_mac_rows(yo, l == 0 ? x : xo, K + 1, a.old_pack + c.w_off[l], OP, o0);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int o = o0 + i;
            if (o >= O) continue;
            if (!last) {
              sm_npg[q.a_off[l + 1] + r * q.sa[l + 1] + o] = c.tanh_act ? tanhf(y[i]) : fmaxf(y[i], 0.f);
              sm_npg[q.da_off[l + 1] + r * q.sa[l + 1] + o] = c.tanh_act ? tanhf(yo[i]) : fmaxf(yo[i], 0.f);
            } else {
              sm_npg[q.d_off[l] + r * q.sd[l] + o] = y[i];
              sm_npg[q.da_off[0] + r * q.sd[l] + o] = yo[i];
            }
          }
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int o = o0 + i;
            if (o >= O) continue;
            if (!last) {
              float* nxt = sm_npg + q.a_off[l + 1] + r * q.sa[l + 1] + o;
              if (MODE == kNpgFvp) {
                sm_npg[q.da_off[l + 1] + r * q.sa[l + 1] + o] = npg_act_grad(c.tanh_act, *nxt) * y[i];
              } else {
                *nxt = c.tanh_act ? tanhf(y[i]) : fmaxf(y[i], 0.f);
              }
            } else {
              sm_npg[q.d_off[l] + r * q.sd[l] + o] = y[i];
            }
          }
        }
      }
      __syncthreads();
    }
    if (MODE == kNpgPrep) {
      for (int l = 1; l < L; ++l) {
        const int w = c.in_dim[l];
        for (int i = threadIdx.x; i < R * w; i += blockDim.x) {
          const int r = i / w, k = i - r * w;
          const long long row = r0 + r;
          if (row < a.n_rows) a.cache[row * q.cache_w + q.cache_off[l] + k] = sm_npg[q.a_off[l] + r * q.sa[l] + k];
        }
      }
      continue;
    }
    // ---- output stage, one thread per row: the cotangent of the last pre-activation and the per-row scalars
    {
      const int sdL = q.sd[L - 1];
      for (int r = threadIdx.x; r < R; r += blockDim.x) {
        const long long src = s_src[r];
        const bool ok = src >= 0;
        float* y = sm_npg + q.d_off[L - 1] + r * sdL;
        float* e = E + r * q.se;
        for (int j = 0; j < A + kNpgExtra; ++j) e[j] = 0.f;
        if (MODE == kNpgGrad) {
          const float ad = ok ? a.adv[src] : 0.f;
          for (int j = 0; j < A; ++j) {
            const float mu = fmaf(y[j], out_scale[j], out_shift[j]);
            const float sd = stdv[j];
            const float z = ok ? (a.act[src * A + j] - mu) / sd : 0.f;
            y[j] = ok ? ad * z / sd * out_scale[j] : 0.f;     // d(adv * LL)/d(pre-activation)
            e[j] = ok ? ad * (z * z - 1.f) : 0.f;             // d(adv * LL)/d(log_std_j)
          }
          e[A] = ok ? 1.f : 0.f;
          e[A + 1] = ad;
        } else if (MODE == kNpgFvp) {
          for (int j = 0; j < A; ++j) {
            const float sd = stdv[j];
            const float dmu = y[j] * out_scale[j];
            y[j] = ok ? dmu * (2.f / (2.f * sd * sd + 1e-8f)) * out_scale[j] : 0.f;
          }
          e[A] = ok ? 1.f : 0.f;
        } else {  // DIAG: surrogate ratio and KL of new vs old per row
          const float* yo = sm_npg + q.da_off[0] + r * sdL;
          float dll = 0.f, kl = 0.f;
          for (int j = 0; j < A; ++j) {
            const float mun = fmaf(y[j], out_scale[j], out_shift[j]);
            const float muo = fmaf(yo[j], out_scale[j], out_shift[j]);
            const float sn = stdv[j], so = a.old_tail[j];
            const float act = ok ? a.act[src * A + j] : 0.f;
            const float zn = (act - mun) / sn, zo = (act - muo) / so;
            dll += -0.5f * zn * zn + 0.5f * zo * zo - (a.ls_new[j] - a.ls_old[j]);
            const float dm = muo - mun;
            kl += (dm * dm + so * so - sn * sn) / (2.f * sn * sn + 1e-8f) + a.ls_new[j] - a.ls_old[j];
          }
          if (ok) {
            e[A] = 1.f;
            e[A + 1] = expf(dll) * a.adv[src];
            e[A + 2] = kl;
          }
        }
      }
    }
    __syncthreads();
    // ---- backward data: delta_{l-1} = act'(a_l) * (W_l^T delta_l)
    for (int l = L - 1; l >= 1 && (MODE == kNpgGrad || MODE == kNpgFvp); --l) {
      const int K = c.in_dim[l], OP = c.out_pad[l], O4 = (c.out_dim[l] + 3) / 4 * 4;
      const int nq = (K + 3) / 4;
      const int units = (R / 32) * nq;
      for (int u = warp; u < units; u += kNpgWarps) {
        const int half = u / nq, k0 = (u - half * nq) * 4;
        const int r = half * 32 + lane;
        float z[4] = {0.f, 0.f, 0.f, 0.f};
        npg_mac_back(z, sm_npg + q.d_off[l] + r * q.sd[l], O4, Wt + c.w_off[l], OP, k0, K);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (k0 + i < K)
            sm_npg[q.d_off[l - 1] + r * q.sd[l - 1] + k0 + i] =
                npg_act_grad(c.tanh_act, sm_npg[q.a_off[l] + r * q.sa[l] + k0 + i]) * z[i];
      }
      __syncthreads();
    }
    // ---- weight / bias gradients: thread-owned 4x4 blocks summed over the tile's rows
    if (MODE == kNpgGrad || MODE == kNpgFvp) {
#pragma unroll
      for (int j = 0; j < kNpgMaxItems; ++j) {
        const int b = threadIdx.x + j * kNpgThreads;
        if (b >= q.blk0[L]) break;
        int l = 0;
        while (b >= q.blk0[l + 1]) ++l;
        const int bl = b - q.blk0[l];
        const int oq = bl / q.kq[l], kq = bl - oq * q.kq[l];
        const float* ap = sm_npg + q.a_off[l] + kq * 4;
        const float* dp = sm_npg + q.d_off[l] + oq * 4;
        const int sa = q.sa[l], sd = q.sd[l];
#pragma unroll 1
        for (int r = 0; r < R; ++r) {
          const float4 x = *reinterpret_cast<const float4*>(ap + r * sa);
          const float4 d = *reinterpret_cast<const float4*>(dp + r * sd);
          const float dv[4] = {d.x, d.y, d.z, d.w}, xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[j][i * 4 + k] = fmaf(dv[i], xv[k], acc[j][i * 4 + k]);
        }
      }
    }
    if (threadIdx.x < A + kNpgExtra)
      for (int r = 0; r < R; ++r) ext += E[r * q.se + threadIdx.x];
  }
  float* part = a.partial + static_cast<long long>(blockIdx.x) * q.pstride;
  if (MODE == kNpgGrad || MODE == kNpgFvp) {
#pragma unroll
    for (int j = 0; j < kNpgMaxItems; ++j) {
      const int b = threadIdx.x + j * kNpgThreads;
      if (b < q.blk0[L]) {
#pragma unroll
        for (int e = 0; e < 16; e += 4)
          *reinterpret_cast<float4*>(part + b * 16 + e) = make_float4(acc[j][e], acc[j][e + 1], acc[j][e + 2], acc[j][e + 3]);
      }
    }
  }
  if (threadIdx.x < A + kNpgExtra) part[q.blk0[L] * 16 + threadIdx.x] = ext;
}

// out[dst[col]] = sum over blocks (fixed order, fp64) of partial[b][col]; dst < 0: column not used.
// mode 0 (gradient): every mapped column.  mode 2 (diagnostics): out[0..2] = the three per-row sums after the
// log_std columns (rows, ratio * advantage, KL).  mode 1 (FVP): out[P] = row count, out[P + 1] = 0 (the advantage
// partials are 0 there); the log_std block of the Fisher is diagonal and the same for every row, so
// out[ls0 + j] = count * 4 s^2 (2 s^2 - eps) / (2 s^2 + eps)^2 * v[ls0 + j] with s the policy std (mjrl's mean_kl,
// eps 1e-8).
__global__ void __launch_bounds__(256)
npg_reduce_kernel(const float* __restrict__ partial, int n_blocks, int pstride, const int* __restrict__ dst,
                  double* __restrict__ out, int mode, int count_col, int ls0, int act_dim, const float* __restrict__ stdv,
                  const double* __restrict__ v, const int* __restrict__ skip) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  if (skip && *skip) return;
  for (int col = blockIdx.x * blockDim.x + threadIdx.x; col < pstride; col += gridDim.x * blockDim.x) {
    int d = dst[col];
    if (mode == 1 && col >= count_col - act_dim && col < count_col) continue;  // log_std: written below
    if (mode == 2) d = (col >= count_col && col < count_col + 3) ? col - count_col : -1;
    if (d < 0) continue;
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += static_cast<double>(partial[static_cast<long long>(b) * pstride + col]);
    out[d] = s;
    if (mode == 1 && col == count_col) {
      for (int j = 0; j < act_dim; ++j) {
        const double s2 = static_cast<double>(stdv[j]) * stdv[j];
        const double h = 4.0 * s2 * (2.0 * s2 - 1e-8) / ((2.0 * s2 + 1e-8) * (2.0 * s2 + 1e-8));
        out[ls0 + j] = s * h * v[ls0 + j];
      }
    }
  }
}

// direction (fp64, mjrl flat order) -> fp32 pack layout for the FVP kernel; pack_of[i] = pack index of flat entry i
// (-1 for log_std entries)
__global__ void npg_to_pack_kernel(const double* __restrict__ v, const int* __restrict__ pack_of, int P,
                                   float* __restrict__ vpack, const int* __restrict__ skip) {
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  if (skip && *skip) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x)
    if (pack_of[i] >= 0) vpack[pack_of[i]] = static_cast<float>(v[i]);
}

// ---- CG bookkeeping (one CTA, fp64, fixed-order reductions) -------------------------------------------------------
struct NpgScalars {
  double rdotr;        // r.r of the current residual
  double gx;           // g.x after the solve
  double alpha;        // step size of the last apply
  double n_grad;       // rows of the gradient (global after the caller's all-reduce)
  double surr_before;  // mean advantage
  double iters;        // CG iterations run
  int done;            // CG converged (rdotr < 1e-10): remaining iterations are no-ops
  int pad;
};

__device__ double npg_block_sum(double v, double* sh) {
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < (blockDim.x + 31) / 32; ++w) t += sh[w];
  return t;
}

// op 0: start from the gradient sums g_sum [P + 2] (P entries, row count, advantage sum): g = g_sum / count, x = 0,
//       r = p = g (cg_solve.py: x = 0, r = b, p = r).
// op 1: one cg_solve iteration given the Fisher sums z_sum [P + 1]: z = z_sum / count + damping p; v = rdotr / p.z;
//       x += v p; r -= v z; p = r + (r.r / rdotr) p; done once rdotr < 1e-10.
__global__ void __launch_bounds__(kNpgCgThreads)
npg_cg_kernel(int op, const double* __restrict__ sums, int P, double damping, double* __restrict__ g,
              double* __restrict__ x, double* __restrict__ r, double* __restrict__ p, NpgScalars* __restrict__ s,
              int* __restrict__ skip) {
  __shared__ double sh[32];
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  if (op == 0) {
    const double cnt = sums[P];
    const double inv = cnt > 0.0 ? 1.0 / cnt : 0.0;
    double rr = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
      const double gi = sums[i] * inv;
      g[i] = gi; x[i] = 0.0; r[i] = gi; p[i] = gi;
      rr += gi * gi;
    }
    rr = npg_block_sum(rr, sh);
    if (threadIdx.x == 0) {
      s->rdotr = rr;
      s->n_grad = cnt;
      s->surr_before = sums[P + 1] * inv;
      s->iters = 0.0;
      s->done = rr == 0.0 ? 1 : 0;   // a zero gradient: nothing to solve
      s->gx = 0.0;
      *skip = s->done;
    }
    return;
  }
  if (s->done) return;
  const double cnt = sums[P];
  const double inv = cnt > 0.0 ? 1.0 / cnt : 0.0;
  double pz = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) pz += p[i] * (sums[i] * inv + damping * p[i]);
  pz = npg_block_sum(pz, sh);
  const double rdotr = s->rdotr;
  const double v = rdotr / pz;
  double rr = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    const double zi = sums[i] * inv + damping * p[i];
    x[i] += v * p[i];
    r[i] -= v * zi;
    rr += r[i] * r[i];
  }
  rr = npg_block_sum(rr, sh);
  const double mu = rr / rdotr;
  for (int i = threadIdx.x; i < P; i += blockDim.x) p[i] = r[i] + mu * p[i];
  __syncthreads();
  if (threadIdx.x == 0) {
    s->rdotr = rr;
    s->iters += 1.0;
    if (rr < 1e-10) { s->done = 1; *skip = 1; }
  }
}

// Flat entry i (mjrl order) of value t into the policy: pack_of[i] >= 0 is its place in the pack, else it is
// log_std[i - ls0] and goes to std[i - ls0] = float(exp(double(t))), exactly as simstep_load_policy stores it.
__device__ __forceinline__ void policy_store_flat(int i, float t, const int* __restrict__ pack_of, int ls0,
                                                  float* __restrict__ pack, float* __restrict__ stdv) {
  if (pack_of[i] >= 0) pack[pack_of[i]] = t;
  else stdv[i - ls0] = static_cast<float>(exp(static_cast<double>(t)));
}

// theta (fp32, mjrl flat order) -> pack (transposed weights, biases) and tail std (policy_store_flat).  APPLY
// (x != null) first forms the NPG step:
//   alpha = const_lr ? lr : sqrt(|delta / (g.x + 1e-10)|),  theta <- float(theta + alpha x),
//   log_std <- max(log_std, min_log_std) (MLP.set_param_values), and keeps the previous parameters in old_* for the
//   diagnostics pass.
__global__ void __launch_bounds__(kNpgCgThreads)
npg_write_kernel(float* __restrict__ theta, const int* __restrict__ pack_of, int P, int ls0, int act_dim, int tail_std0,
                 float* __restrict__ pack, int pack_floats, float* __restrict__ tail, const double* __restrict__ g,
                 const double* __restrict__ x, double step, int const_lr, float min_log_std,
                 float* __restrict__ old_pack, float* __restrict__ old_theta, float* __restrict__ old_std,
                 NpgScalars* __restrict__ s, int* __restrict__ skip) {
  __shared__ double sh[32];
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  double alpha = 0.0;
  if (x) {
    for (int i = threadIdx.x; i < pack_floats; i += blockDim.x) old_pack[i] = pack[i];
    for (int j = threadIdx.x; j < act_dim; j += blockDim.x) old_std[j] = tail[tail_std0 + j];
    double gx = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) gx += g[i] * x[i];
    gx = npg_block_sum(gx, sh);
    alpha = const_lr ? step : sqrt(fabs(step / (gx + 1e-10)));
    if (threadIdx.x == 0) { s->gx = gx; s->alpha = alpha; }
    __syncthreads();  // old_pack is complete before pack is overwritten
  }
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    float t = theta[i];
    if (x) {
      old_theta[i] = t;
      t = static_cast<float>(static_cast<double>(t) + alpha * x[i]);
      if (i >= ls0) t = fmaxf(t, min_log_std);
      theta[i] = t;
    }
    policy_store_flat(i, t, pack_of, ls0, pack, tail + tail_std0);
  }
  if (x && threadIdx.x == 0) *skip = 0;
}

}  // namespace simstep
