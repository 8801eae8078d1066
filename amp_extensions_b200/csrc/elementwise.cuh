// HBM-bound kernels around the ensemble GEMMs: input normalisation, the fused
// next-state / discrepancy / termination kernel, RFF operand packing and small
// reductions.  All row-parallel, coalesced, no atomics on the data path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gemm_tcgen05.cuh"
#include "../../include/simstep.h"

namespace simstep {

// ---- operand packing -----------------------------------------------------

struct PackSegs {
  int n;
  int src0[SIMSTEP_MAX_HIDDEN + 2];
  int width[SIMSTEP_MAX_HIDDEN + 2];
  int dst0[SIMSTEP_MAX_HIDDEN + 2];
};

// dst[o][dst0+i] = cvt(src[o][src0+i]) for every segment, dst pre-zeroed.
// One block row per output feature; used once at load time.
template <typename E>
__global__ void pack_weight_kernel(const float* __restrict__ src, int src_pitch, int rows,
                                   typename E::storage* __restrict__ dst, long long dst_pitch, PackSegs segs,
                                   int mode /*0 value, 1 hi, 2 lo, 3 raw fp32 bits (training master copy)*/) {
  const int o = blockIdx.x;
  if (o >= rows) return;
  for (int s = 0; s < segs.n; ++s) {
    for (int i = threadIdx.x; i < segs.width[s]; i += blockDim.x) {
      const float v = src[size_t(o) * src_pitch + segs.src0[s] + i];
      float out = v;
      if (mode == 2) out = v - static_cast<float>(E::cvt(v));
      dst[size_t(o) * dst_pitch + segs.dst0[s] + i] = mode == 3 ? static_cast<typename E::storage>(v) : E::cvt(out);
    }
  }
}

template <typename T>
struct Pair;
template <>
struct Pair<float> { using type = float2; };
template <>
struct Pair<__half> { using type = __half2; };
template <>
struct Pair<__nv_bfloat16> { using type = __nv_bfloat162; };

template <typename E>
__device__ __forceinline__ typename Pair<typename E::storage>::type make_pair_cvt(float a, float b) {
  typename Pair<typename E::storage>::type p;
  p.x = E::cvt(a);
  p.y = E::cvt(b);
  return p;
}

// x = [(s - mean_s)/scale_s, (a - mean_a)/scale_a, 0...]  (reference
// milo/milo/dynamics.py:225-230) written in the GEMM operand format.  Rows in
// [n_rows, rows_pad) are zero-filled so padded tiles stay finite.  One block
// walks rows; each thread owns two adjacent columns (XP is even) and stores
// them as one packed pair.  VEC: S and A are even and both sources 8-byte
// aligned, so a column pair never straddles the state / action boundary and is
// read with one 8-byte load.  The kernel was issue-bound (ncu: 16 M warp
// instructions for 61 MB of traffic), hence the per-thread source pointer,
// the hoisted reciprocal scale and the pointer-stepped row loop.
constexpr int kPrepThreads = 128;
#ifndef SIMSTEP_PREP_ROWS
#define SIMSTEP_PREP_ROWS 4
#endif
constexpr int kPrepRows = SIMSTEP_PREP_ROWS;
template <typename E, bool VEC>
__global__ void __launch_bounds__(kPrepThreads)
prep_input_kernel(const float* __restrict__ state, const float* __restrict__ action, int S, int A, int XP,
                  long long n_rows, long long rows_pad,
                  const float* __restrict__ tf /* mean_s|scale_s|mean_a|scale_a or null */,
                  typename E::storage* __restrict__ x, const float* __restrict__ w_src, float* __restrict__ w_dst,
                  int w_len, unsigned long long* __restrict__ saturated) {
  using P = typename Pair<typename E::storage>::type;
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  // the step's cost weights ride along: block 0 stages w into the zero-padded vector the RFF epilogue reads
  if (w_src != nullptr && blockIdx.x == 0)
    for (int i = threadIdx.x; i < w_len; i += kPrepThreads) w_dst[i] = w_src[i];
  const long long stride = gridDim.x;
  for (int c0 = 2 * threadIdx.x; c0 < XP; c0 += 2 * kPrepThreads) {
    // per-column constants hoisted out of the row loop
    float mean[2] = {0.f, 0.f}, rscale[2] = {1.f, 1.f};
    const float* col_ptr[2] = {nullptr, nullptr};  // null: zero padding
    long long pitch[2] = {0, 0};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int col = c0 + i;
      if (col < S) {
        col_ptr[i] = state + col;
        pitch[i] = S;
        if (tf) { mean[i] = tf[col]; rscale[i] = 1.f / tf[S + col]; }
      } else if (col < S + A) {
        col_ptr[i] = action + (col - S);
        pitch[i] = A;
        if (tf) { mean[i] = tf[2 * S + col - S]; rscale[i] = 1.f / tf[2 * S + A + col - S]; }
      }
    }
    // kPrepRows rows per trip: all their loads are issued before the first is used
    for (long long row0 = blockIdx.x; row0 < rows_pad; row0 += stride * kPrepRows) {
      float v[kPrepRows][2];
#pragma unroll
      for (int r = 0; r < kPrepRows; ++r) {
        const long long row = row0 + r * stride;
        v[r][0] = v[r][1] = 0.f;
        if (row < n_rows) {
          if (VEC) {
            if (col_ptr[0] != nullptr) {
              const float2 t = *reinterpret_cast<const float2*>(col_ptr[0] + row * pitch[0]);
              v[r][0] = t.x;
              v[r][1] = t.y;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 2; ++i)
              if (col_ptr[i] != nullptr) v[r][i] = col_ptr[i][row * pitch[i]];
          }
        }
      }
#pragma unroll
      for (int r = 0; r < kPrepRows; ++r) {
        const long long row = row0 + r * stride;
        if (row < rows_pad) {
          float o[2] = {0.f, 0.f};
          if (row < n_rows) {
#pragma unroll
            for (int i = 0; i < 2; ++i)
              if (col_ptr[i] != nullptr) o[i] = (v[r][i] - mean[i]) * rscale[i];
            // fp16 operands saturate at 65 504 where the fp32 reference carries on (a dataset column with scale
            // 1e-8, datasets.py:35-40, and a state that drifted): count it, the host can ask (rare path)
            if (E::kKind == 1 && E::kFmt == 0 && saturated != nullptr &&
                (fabsf(o[0]) > 65504.f || fabsf(o[1]) > 65504.f))
              atomicAdd(saturated, 1ull);
          }
          *reinterpret_cast<P*>(x + row * XP + c0) = make_pair_cvt<E>(o[0], o[1]);
        }
      }
    }
  }
}

// RFF operand rows: concatenation of up to three fp32 sources, optionally as
// [hi | lo | hi] operand triple (see simstep_load_rff).
struct RffSrc {
  int n;
  const float* ptr[3];   // first element of the segment in row 0
  int width[3];          // columns taken from the segment
  int pitch[3];          // floats between consecutive rows of the segment's source
  int dst0[3];           // operand column of the segment's first element (segments may leave gaps: zero padding)
};

// out row = [hi(x) | lo(x)] (split) or [hi(x)] with x the concatenation of the sources zero-padded to RK; the
// GEMM re-reads the hi block for the third product (x_hi * W_lo), so it is stored once.
template <typename E>
__global__ void __launch_bounds__(kPrepThreads)
rff_pack_kernel(RffSrc src, int RK, int split, int pitch, long long n_rows, long long rows_pad,
                typename E::storage* __restrict__ out) {
  using P = typename Pair<typename E::storage>::type;
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  for (int c0 = 2 * threadIdx.x; c0 < RK; c0 += 2 * kPrepThreads) {
    const float* base[2] = {nullptr, nullptr};
    int spitch[2] = {0, 0};
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int c = c0 + i;
#pragma unroll
      for (int k = 0; k < 3; ++k)
        if (k < src.n && c >= src.dst0[k] && c < src.dst0[k] + src.width[k]) {
          base[i] = src.ptr[k] + (c - src.dst0[k]);
          spitch[i] = src.pitch[k];
        }
    }
    for (long long row = blockIdx.x; row < rows_pad; row += gridDim.x) {
      float v[2] = {0.f, 0.f};
      if (row < n_rows) {
        if (base[0]) v[0] = base[0][row * spitch[0]];
        if (base[1]) v[1] = base[1][row * spitch[1]];
      }
      const P hi = make_pair_cvt<E>(v[0], v[1]);
      typename E::storage* orow = out + row * pitch;
      *reinterpret_cast<P*>(orow + c0) = hi;
      if (split)
        *reinterpret_cast<P*>(orow + RK + c0) =
            make_pair_cvt<E>(v[0] - static_cast<float>(hi.x), v[1] - static_cast<float>(hi.y));
    }
  }
}

// ---- fused next-state / discrepancy / termination kernel -------------------

struct TermConst {
  int horizon;
  int enable_velocity_check;
  int vel_offset;
  float vel_threshold;
  float vel_inv_divisor;
  int record_all_world;
  int record_world_root_pos;
  int n_bodies;
  int pos_dim;
  int body_offset[SIMSTEP_MAX_BODIES];
  int body_shape[SIMSTEP_MAX_BODIES];
  float body_radius[SIMSTEP_MAX_BODIES];      // 0.5*Param0
  float body_half_height[SIMSTEP_MAX_BODIES]; // 0.5*Param1
};

constexpr int kPostWarps = 8;
constexpr int kPostMaxElems = 256;  // supports S <= 256

template <int VEC>
struct PostVec;
template <>
struct PostVec<1> {
  using type = float;
  __device__ static __forceinline__ float zero() { return 0.f; }
  __device__ static __forceinline__ float nan() { return __int_as_float(0x7fc00000); }
  __device__ static __forceinline__ float sub_sq(float a, float b, float acc) { const float t = a - b; return fmaf(t, t, acc); }
  __device__ static __forceinline__ float add(float a, float b) { return a + b; }
  __device__ static __forceinline__ bool vel_over(float v, int j, int off, float inv_div, float thr) {
    return j >= off && fabsf(v * inv_div) > thr;
  }
};
template <>
struct PostVec<2> {
  using type = float2;
  __device__ static __forceinline__ float2 zero() { return make_float2(0.f, 0.f); }
  __device__ static __forceinline__ float2 nan() { return make_float2(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000)); }
  __device__ static __forceinline__ float sub_sq(float2 a, float2 b, float acc) {
    const float t0 = a.x - b.x, t1 = a.y - b.y;
    return fmaf(t1, t1, fmaf(t0, t0, acc));
  }
  __device__ static __forceinline__ float2 add(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
  __device__ static __forceinline__ bool vel_over(float2 v, int j, int off, float inv_div, float thr) {
    return (j >= off && fabsf(v.x * inv_div) > thr) || (j + 1 >= off && fabsf(v.y * inv_div) > thr);
  }
};

// RFF operand row of the fused step: [hi(s) | 0 | hi(s') | 0][lo(s) | 0 | lo(s') | 0] (see rff_pack_kernel; s' starts at
// column col2 = S rounded up to 8, so both halves can be written with 16-byte stores), written by
// the same warp that produced s'.  prec: SIMSTEP_PREC_*; out == nullptr: not fused.
struct PostRff {
  void* out;
  int prec;
  int RK;
  int split;
  int col2;  // operand column of s' (s starts at column 0)
  int pitch; // elements per operand row (2 RK when the rows were allocated for hi/lo pairs, whether or not split is on)
};

template <typename E>
__device__ __forceinline__ void post_rff_store(const PostRff& r, long long row, int col, float2 v) {
  using T = typename E::storage;
  using P = typename Pair<T>::type;
  T* orow = static_cast<T*>(r.out) + row * r.pitch;
  const P hi = make_pair_cvt<E>(v.x, v.y);
  *reinterpret_cast<P*>(orow + col) = hi;
  if (r.split)
    *reinterpret_cast<P*>(orow + r.RK + col) =
        make_pair_cvt<E>(v.x - static_cast<float>(hi.x), v.y - static_cast<float>(hi.y));
}

// One warp per env row (reference: sim_env.py:140-173 for the step and the
// termination test, dynamics.py:134-143 for the discrepancy).
//   delta  [NM][delta_rows][SP] fp32 workspace of the final GEMM, row = chunk-local
//   state  [E][S], next_state [E][S] (may alias state)
// VEC = 2 when S is even: every row then starts 8-byte aligned and lanes move float2.
// One env row, one warp: the body of post_step_kernel.  srow: this warp's shared-memory row of (S + 3) & ~3 floats.
template <int NM, int VEC>
__device__ __forceinline__ void post_row_warp(const float* __restrict__ delta, long long delta_rows, int SP,
                                              const float* state, const int32_t* __restrict__ member,
                                              int32_t* num_steps, int S, long long row, float* next_state,
                                              float* __restrict__ disc, uint8_t* __restrict__ done,
                                              const TermConst& tc, const PostRff& rff, float* srow, int lane) {
  using V = typename PostVec<VEC>::type;
  constexpr int kPerLane = kPostMaxElems / (32 * VEC);
  constexpr int NP = NM * (NM - 1) / 2;
  const int nvec = S / VEC;
  V d[NM][kPerLane];
#pragma unroll
  for (int m = 0; m < NM; ++m) {
    const V* drow = reinterpret_cast<const V*>(delta + (static_cast<long long>(m) * delta_rows + row) * SP);
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) {
      const int j = lane + 32 * i;
      d[m][i] = (j < nvec) ? __ldg(drow + j) : PostVec<VEC>::zero();
    }
  }
  V sv[kPerLane];
  if (next_state != nullptr) {
    const V* srow_g = reinterpret_cast<const V*>(state + row * S);
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) {
      const int j = lane + 32 * i;
      sv[i] = (j < nvec) ? srow_g[j] : PostVec<VEC>::zero();
    }
  }

  if (disc != nullptr) {
    float acc[NP > 0 ? NP : 1];
    int p = 0;
#pragma unroll
    for (int a = 0; a < NM; ++a) {
#pragma unroll
      for (int b = a + 1; b < NM; ++b) {
        float s2 = 0.f;
#pragma unroll
        for (int i = 0; i < kPerLane; ++i) s2 = PostVec<VEC>::sub_sq(d[a][i], d[b][i], s2);
        acc[p++] = s2;
      }
    }
    float best = 0.f;
#pragma unroll
    for (int k = 0; k < NP; ++k) {
      float s2 = acc[k];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, off);
      // NaN must propagate like torch.max does
      if (s2 != s2) best = s2;
      else if (best == best && s2 > best) best = s2;
    }
    if (lane == 0) disc[row] = sqrtf(best);
  }

  if (next_state != nullptr) {
    const int mem = member ? member[row] : 0;
    V nxt[kPerLane];
    V* nrow_g = reinterpret_cast<V*>(next_state + row * S);
    V* srow_v = reinterpret_cast<V*>(srow);
#pragma unroll
    for (int i = 0; i < kPerLane; ++i) {
      const int j = lane + 32 * i;
      V dm = PostVec<VEC>::nan();  // a member index outside [0, N) (the reference raises IndexError): NaN next state
#pragma unroll
      for (int m = 0; m < NM; ++m) dm = (m == mem) ? d[m][i] : dm;
      nxt[i] = PostVec<VEC>::add(sv[i], dm);
      if (j < nvec) {
        nrow_g[j] = nxt[i];
        srow_v[j] = nxt[i];
      }
    }
    if constexpr (VEC == 2) {
      if (rff.out != nullptr) {  // cost features' operand rows for input_type 'ss' (linear_cost.py:119)
#pragma unroll
        for (int i = 0; i < kPerLane; ++i) {
          const int j = lane + 32 * i;
          if (j < nvec) {
            if (rff.prec == SIMSTEP_PREC_FP16) {
              post_rff_store<ElemF16>(rff, row, 2 * j, sv[i]);
              post_rff_store<ElemF16>(rff, row, rff.col2 + 2 * j, nxt[i]);
            } else if (rff.prec == SIMSTEP_PREC_TF32) {
              post_rff_store<ElemTF32>(rff, row, 2 * j, sv[i]);
              post_rff_store<ElemTF32>(rff, row, rff.col2 + 2 * j, nxt[i]);
            } else {
              post_rff_store<ElemBF16>(rff, row, 2 * j, sv[i]);
              post_rff_store<ElemBF16>(rff, row, rff.col2 + 2 * j, nxt[i]);
            }
          }
        }
      }
    }
    int steps = 0;
    if (num_steps != nullptr) {
      steps = num_steps[row] + 1;
      if (lane == 0) num_steps[row] = steps;
    }
    if (done != nullptr) {
      __syncwarp();
      bool flag = false;
      if (lane < tc.n_bodies) {
        const int off = tc.body_offset[lane];
        const int shape = tc.body_shape[lane];
        float y = srow[off + 1];
        if (!(tc.record_all_world || (lane == 0 && tc.record_world_root_pos))) y += srow[0];
        const float lim = tc.body_radius[lane] + 0.0001f;
        if (shape == SIMSTEP_SHAPE_SPHERE) {
          flag = y <= lim;
        } else if (shape == SIMSTEP_SHAPE_CAPSULE) {
          const float cap = tc.body_half_height[lane] * srow[off + tc.pos_dim + 1];
          flag = (y + cap <= lim) || (y - cap <= lim);
        }
      }
      if (tc.enable_velocity_check) {
#pragma unroll
        for (int i = 0; i < kPerLane; ++i) {
          const int j = (lane + 32 * i) * VEC;  // first element of this lane's slot
          if (j < S) flag = flag || PostVec<VEC>::vel_over(nxt[i], j, tc.vel_offset, tc.vel_inv_divisor, tc.vel_threshold);
        }
      }
      const bool any = __any_sync(0xffffffffu, flag);
      if (lane == 0) done[row] = (any || (num_steps != nullptr && steps >= tc.horizon)) ? 1 : 0;
      __syncwarp();
    }
  }
}

template <int NM, int VEC>
__global__ void __launch_bounds__(kPostWarps * 32, NM <= 4 ? 3 : 2)
post_step_kernel(const float* __restrict__ delta, long long delta_rows, int SP, const float* state,
                 const int32_t* __restrict__ member, int32_t* num_steps, int S, long long n_rows,
                 float* next_state, float* __restrict__ disc, uint8_t* __restrict__ done, const TermConst tc,
                 const PostRff rff) {
  extern __shared__ float sm_rows[];  // [kPostWarps][S]
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  float* srow = sm_rows + size_t(wib) * ((S + 3) & ~3);
  const long long warp_global = blockIdx.x * static_cast<long long>(kPostWarps) + wib;
  const long long n_warps = static_cast<long long>(gridDim.x) * kPostWarps;
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();
  for (long long row = warp_global; row < n_rows; row += n_warps)
    post_row_warp<NM, VEC>(delta, delta_rows, SP, state, member, num_steps, S, row, next_state, disc, done, tc,
                                  rff, srow, lane);
}

// delta workspace -> dense [NM][E][S] rows (DynamicsModel.forward's return value)
static __global__ void extract_delta_kernel(const float* __restrict__ ws, long long ws_rows, int SP, int NM, int S,
                                     long long n_rows, float* __restrict__ out, long long out_rows,
                                     long long out_row0) {
  const long long total = static_cast<long long>(NM) * n_rows * S;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int j = static_cast<int>(idx % S);
    const long long t = idx / S;
    const long long row = t % n_rows;
    const int m = static_cast<int>(t / n_rows);
    out[(static_cast<long long>(m) * out_rows + out_row0 + row) * S + j] =
        ws[(static_cast<long long>(m) * ws_rows + row) * SP + j];
  }
}

// ---- reductions ------------------------------------------------------------

// column sums of a [n_rows][D] fp32 matrix, fp64 accumulate, two passes so the
// result does not depend on scheduling: partial[b][d] then final.
static __global__ void colsum_partial_kernel(const float* __restrict__ x, long long n_rows, int D, int rows_per_block,
                                      double* __restrict__ partial) {
  const long long r0 = static_cast<long long>(blockIdx.x) * rows_per_block;
  const long long r1 = min(r0 + rows_per_block, n_rows);
  for (int dcol = threadIdx.x; dcol < D; dcol += blockDim.x) {
    double s = 0.0;
    for (long long r = r0; r < r1; ++r) s += static_cast<double>(x[r * D + dcol]);
    partial[static_cast<long long>(blockIdx.x) * D + dcol] = s;
  }
}
static __global__ void colsum_final_kernel(const double* __restrict__ partial, int n_blocks, int D, double* __restrict__ out,
                                    int accumulate) {
  for (int dcol = blockIdx.x * blockDim.x + threadIdx.x; dcol < D; dcol += gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += partial[static_cast<long long>(b) * D + dcol];
    out[dcol] = accumulate ? out[dcol] + s : s;
  }
}

// out[0] = max, out[1] = sum; single block, deterministic.
static __global__ void reduce_max_sum_kernel(const float* __restrict__ x, long long n, double* __restrict__ out) {
  __shared__ double s_sum[32];
  __shared__ float s_max[32];
  double sum = 0.0;
  float mx = -INFINITY;
  bool nan = false;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) {
    const float v = x[i];
    sum += v;
    nan = nan || (v != v);
    mx = fmaxf(mx, v);
  }
  if (nan) mx = NAN;
  for (int off = 16; off > 0; off >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, off);
    const float o = __shfl_xor_sync(0xffffffffu, mx, off);
    mx = (mx != mx || o != o) ? NAN : fmaxf(mx, o);
  }
  if ((threadIdx.x & 31) == 0) {
    s_sum[threadIdx.x >> 5] = sum;
    s_max[threadIdx.x >> 5] = mx;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0;
    float tm = -INFINITY;
    for (int w = 0; w < (blockDim.x + 31) / 32; ++w) {
      ts += s_sum[w];
      tm = (tm != tm || s_max[w] != s_max[w]) ? NAN : fmaxf(tm, s_max[w]);
    }
    out[0] = tm;
    out[1] = ts;
  }
}

}  // namespace simstep
