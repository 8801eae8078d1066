// Fused next-state / discrepancy / termination / cost-operand kernel, TMA-staged (reference:
// gym-simenv/gym_simenv/envs/sim_env.py:140-173 for the step and the termination test, milo/milo/dynamics.py:134-143
// for the discrepancy, milo/milo/linear_cost.py:115-126 for the [s; s'] cost input).
//
// The kernel is HBM-bound (5.4 KB read, 2.9 KB written per env at N = 4), so it is organised around keeping bytes
// in flight rather than around arithmetic: a persistent grid of one block per SM, every team of two warps an
// independent producer/consumer pipeline over PAIRS of env rows.  One lane issues 1-D bulk copies (cp.async.bulk,
// completion on the team's own mbarriers) of the pair's state rows and of its N member-delta rows into a private
// ring of shared-memory stages, up to `stages` pairs ahead; each warp then computes one row from shared memory
// (conflict-free 8-byte lanes) and writes its outputs with coalesced stores.  No block-level synchronisation after
// the barrier set-up.
//
// Pairs, because a state row is 904 bytes: two consecutive rows are one 16-byte aligned, 16-byte granular span,
// which is what a bulk copy needs.  The delta workspace has a 912-byte row pitch (S rounded up to 4 floats) for
// the same reason.  An odd trailing row is staged with plain loads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "elementwise.cuh"
#include "ptx.cuh"

namespace simstep {

// 10 rings of two warps, 2 stages each: measured (B200, 40 000 rows, 4 members) 48.0 us against 49.3 us for 8 x 2,
// 55.0 us for 8 x 3 and 60.1 us for 6 x 4 - more warps beat deeper rings
constexpr int kPostTmaMaxWarps = 20;
constexpr int kPostTmaLaunchWarps = 20;  // launch bound
constexpr int kPostTmaMaxStages = 2;
constexpr int kPostTmaSmemBudget = 216 * 1024;

struct PostTmaPlan {
  int rings;   // two-warp teams per block, one ring of stages each
  int stages;
  int stage_bytes;
  size_t smem;
  bool ok;
};

// Host side: rings per block and ring depth such that the rings fit in shared memory.
inline PostTmaPlan post_tma_plan(int S, int DP, int NM) {
  PostTmaPlan p{};
  p.stage_bytes = 2 * S * 4 + NM * 2 * DP * 4;
  p.rings = kPostTmaMaxWarps / 2;
  p.stages = kPostTmaMaxStages;
  while (p.rings * p.stages * p.stage_bytes > kPostTmaSmemBudget) {
    if (p.stages > 2) --p.stages;
    else if (p.rings > 1) --p.rings;
    else break;
  }
  p.ok = (S % 2 == 0) && (S <= kPostMaxElems) && (DP % 4 == 0) &&
         (p.rings * p.stages * p.stage_bytes <= kPostTmaSmemBudget);
  p.smem = size_t(p.rings) * p.stages * p.stage_bytes + size_t(p.rings) * 2 * p.stages * sizeof(uint64_t);
  return p;
}

template <typename E>
__device__ __forceinline__ void post_tma_rff_store(typename E::storage* orow, int RK, bool split, int col, float2 v) {
  using T = typename E::storage;
  using P = typename Pair<T>::type;
  const P hi = make_pair_cvt<E>(v.x, v.y);
  *reinterpret_cast<P*>(orow + col) = hi;
  if (split)
    *reinterpret_cast<P*>(orow + RK + col) =
        make_pair_cvt<E>(v.x - static_cast<float>(hi.x), v.y - static_cast<float>(hi.y));
}

// Fall-contact constants of the body this lane tests (sim_env.py:175-257), fetched once per kernel.
struct PostLaneBody {
  int off;        // offset of the body's position in the state row, -1: this lane tests nothing
  int shape;
  int normal_y;   // offset of the rotation normal's y component
  float lim;      // 0.5 * Param0 + 1e-4
  float half_h;   // 0.5 * Param1
  bool add_root;  // body position is recorded relative to the root height s[0]
};

__device__ __forceinline__ PostLaneBody post_lane_body(const TermConst& tc, int lane) {
  PostLaneBody b{};
  b.off = -1;
  if (lane < tc.n_bodies) {
    b.off = tc.body_offset[lane];
    b.shape = tc.body_shape[lane];
    b.normal_y = b.off + tc.pos_dim + 1;
    b.lim = tc.body_radius[lane] + 0.0001f;
    b.half_h = tc.body_half_height[lane];
    b.add_root = !(tc.record_all_world || (lane == 0 && tc.record_world_root_pos));
  }
  return b;
}

// max_k sum_lanes v[k] for NP per-lane partial sums, NaN-propagating like torch.max.  Recursive halving: at
// every step a lane hands half of its values to its partner, so NP values cost ~NP shuffles instead of 5 * NP.
template <int NP>
__device__ __forceinline__ float post_max_of_lane_sums(float (&acc)[NP > 0 ? NP : 1], int lane) {
  if constexpr (NP == 0) {
    return 0.f;
  } else {
    constexpr int P = NP <= 1 ? 1 : NP <= 2 ? 2 : NP <= 4 ? 4 : NP <= 8 ? 8 : NP <= 16 ? 16 : 32;
    float v[P];
#pragma unroll
    for (int i = 0; i < P; ++i) v[i] = i < NP ? acc[i] : 0.f;  // squared norms are >= 0: padding never wins the max
    int n = P;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      if (n > 1) {
        n >>= 1;
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < P / 2; ++i) {
          if (i < n) {
            const float send = upper ? v[i] : v[i + n];
            const float keep = upper ? v[i + n] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
          }
        }
      } else {
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
      }
    }
    // the P totals now sit in lanes that differ in the bits consumed by the halving steps (16, 8, ...)
    float best = v[0];
    constexpr int kSteps = P == 1 ? 0 : P == 2 ? 1 : P == 4 ? 2 : P == 8 ? 3 : P == 16 ? 4 : 5;
#pragma unroll
    for (int st = 0; st < kSteps; ++st) {
      const float other = __shfl_xor_sync(0xffffffffu, best, 16 >> st);
      best = (best != best) ? best : ((other != other) ? other : fmaxf(best, other));
    }
    return best;
  }
}

// the member pairs (a, b), a < b, in the order (0,1), (0,2), ..., (1,2), ... as compile-time tables
template <int N>
struct PostPairs {
  static constexpr int kCount = N * (N - 1) / 2;
  int a[kCount > 0 ? kCount : 1];
  int b[kCount > 0 ? kCount : 1];
  constexpr PostPairs() : a{}, b{} {
    int p = 0;
    for (int i = 0; i < N; ++i)
      for (int j = i + 1; j < N; ++j) {
        a[p] = i;
        b[p] = j;
        ++p;
      }
  }
};

// One env row out of a staged pair.  srow: the row's state in shared memory (overwritten with s'), drow0: member
// 0's delta row, member m's row sits m * dstride floats further.  SC: compile-time state width (0: use S).
template <int NM, typename E, int SC>
__device__ __forceinline__ void post_tma_row(float* srow, const float* drow0, int dstride, int S_rt, long long row,
                                             int mem, int steps_in, bool have_steps, float* next_state,
                                             float* __restrict__ disc, uint8_t* __restrict__ done,
                                             int32_t* __restrict__ num_steps, const TermConst& tc,
                                             const PostLaneBody& body, const PostRff& rff, int lane) {
  const int S = SC ? SC : S_rt;
  const int nvec = S >> 1;
  constexpr int kSlots = SC ? (SC / 2 + 31) / 32 : kPostMaxElems / 64;  // float2 slots per lane
  constexpr int kFull = SC ? (SC / 2) / 32 : 0;                           // slots every lane owns
  constexpr int NP = NM * (NM - 1) / 2;
  bool in[kSlots];
#pragma unroll
  for (int i = 0; i < kSlots; ++i) in[i] = (i < kFull) || (lane + 32 * i < nvec);

  float2 d[NM][kSlots];
  float2 sv[kSlots];
  const float2* s2 = reinterpret_cast<const float2*>(srow) + lane;
  const float2* d2 = reinterpret_cast<const float2*>(drow0) + lane;
  const int dstride2 = dstride >> 1;
#pragma unroll
  for (int i = 0; i < kSlots; ++i) {
#pragma unroll
    for (int m = 0; m < NM; ++m) d[m][i] = in[i] ? d2[m * dstride2 + 32 * i] : make_float2(0.f, 0.f);
    sv[i] = in[i] ? s2[32 * i] : make_float2(0.f, 0.f);
  }

  if (disc != nullptr) {
    float acc[NP > 0 ? NP : 1];
    const float2 neg1 = make_float2(-1.f, -1.f);
    // one flat loop over the member pairs (indices are compile-time after unrolling: a nested a/b loop is left
    // partly rolled at N = 8 and drags the delta rows into local memory)
    constexpr PostPairs<NM> pairs{};
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const int a = pairs.a[p], b = pairs.b[p];
      float2 q = make_float2(0.f, 0.f);  // packed fp32 pairs: one issue slot per two elements
#pragma unroll
      for (int i = 0; i < kSlots; ++i) {
        const float2 t = __ffma2_rn(d[b][i], neg1, d[a][i]);  // a - b, exactly
        q = __ffma2_rn(t, t, q);
      }
      acc[p] = q.x + q.y;
    }
    const float best = post_max_of_lane_sums<NP>(acc, lane);
    if (lane == 0) disc[row] = sqrtf(best);
  }

  if (next_state != nullptr) {
    float2 nxt[kSlots];
    float2* nrow_g = reinterpret_cast<float2*>(next_state + row * S) + lane;
    // the active member's row (sim_env.py:157); an index outside [0, N) (the reference raises IndexError) makes the
    // row's next state NaN instead of reading another env's deltas
    const bool mem_ok = mem >= 0 && mem < NM;
    const float2* dm2 = d2 + (mem_ok ? mem : 0) * dstride2;
    const float qnan = __int_as_float(0x7fc00000);
#pragma unroll
    for (int i = 0; i < kSlots; ++i) {
      if (in[i]) {
        nxt[i] = mem_ok ? __fadd2_rn(sv[i], dm2[32 * i]) : make_float2(qnan, qnan);
        nrow_g[32 * i] = nxt[i];
        const_cast<float2*>(s2)[32 * i] = nxt[i];
      } else {
        nxt[i] = make_float2(0.f, 0.f);
      }
    }
    if (rff.out != nullptr) {  // cost features' operand row for input_type 'ss' (linear_cost.py:119)
      using T = typename E::storage;
      T* orow = static_cast<T*>(rff.out) + row * rff.pitch + 2 * lane;
#pragma unroll
      for (int i = 0; i < kSlots; ++i) {
        if (in[i]) {
          post_tma_rff_store<E>(orow, rff.RK, rff.split != 0, 64 * i, sv[i]);
          post_tma_rff_store<E>(orow, rff.RK, rff.split != 0, rff.col2 + 64 * i, nxt[i]);
        }
      }
    }
    const int steps = steps_in + 1;
    if (have_steps && lane == 0) num_steps[row] = steps;
    if (done != nullptr) {
      __syncwarp();
      bool flag = false;
      if (body.off >= 0) {
        float y = srow[body.off + 1];
        if (body.add_root) y += srow[0];
        if (body.shape == SIMSTEP_SHAPE_SPHERE) {
          flag = y <= body.lim;
        } else if (body.shape == SIMSTEP_SHAPE_CAPSULE) {
          const float cap = body.half_h * srow[body.normal_y];
          flag = (y + cap <= body.lim) || (y - cap <= body.lim);
        }
      }
      if (tc.enable_velocity_check) {
#pragma unroll
        for (int i = 0; i < kSlots; ++i) {
          const int j = (lane + 32 * i) * 2;
          if (in[i]) flag = flag || PostVec<2>::vel_over(nxt[i], j, tc.vel_offset, tc.vel_inv_divisor, tc.vel_threshold);
        }
      }
      const bool any = __any_sync(0xffffffffu, flag);
      if (lane == 0) done[row] = (any || (have_steps && steps >= tc.horizon)) ? 1 : 0;
    }
  }
}

// delta [NM][delta_rows][DP] fp32 (16-byte aligned, DP % 4 == 0); state / next_state [E][S] fp32, S even, state
// 16-byte aligned, next_state 8-byte aligned (it may alias state: a row is read and written by one warp only).
//
// Block = `rings` teams of two warps.  A team owns one ring of `stages` shared-memory stages; its warp 0 is also
// the producer (lane 0 issues the bulk copies of a pair of rows), warp r consumes row r of every staged pair.
// full[stage] completes on the copies' bytes; empty[stage] collects one arrival per consumer warp before the
// producer overwrites the stage.  Two warps per ring double the warps that hide instruction latency for the same
// bytes in flight.
template <int NM, typename E, int SC>
__global__ void __launch_bounds__(kPostTmaLaunchWarps * 32, 1)
post_step_tma_kernel(const float* __restrict__ delta, long long delta_rows, int DP, const float* state,
                     const int32_t* __restrict__ member, int32_t* num_steps, int S, long long n_rows,
                     float* next_state, float* __restrict__ disc, uint8_t* __restrict__ done,
                     const TermConst tc, const PostRff rff, int stages, int reverse) {
  if (SC) S = SC;
  extern __shared__ __align__(128) uint8_t sm_post[];
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int rings = blockDim.x >> 6;
  const int team = wib >> 1;
  const int trank = wib & 1;
  const int state_bytes = 2 * S * 4;
  const int delta_bytes = 2 * DP * 4;
  const int stage_bytes = state_bytes + NM * delta_bytes;
  uint8_t* ring = sm_post + size_t(team) * stages * stage_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(sm_post + size_t(rings) * stages * stage_bytes) + team * 2 * stages;
  uint64_t* empty = full + stages;
  if (trank == 0 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      ptx::mbar_init(&full[s], 1);
      ptx::mbar_init(&empty[s], 2);
    }
    ptx::fence_barrier_init();
  }
  const PostLaneBody body = post_lane_body(tc, lane);
  __syncthreads();
  // everything above overlaps the tail of the final-layer GEMM; its deltas are read from here on
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();

  const long long n_pairs = (n_rows + 1) >> 1;
  const long long t_global = blockIdx.x * static_cast<long long>(rings) + team;
  const long long t_total = static_cast<long long>(gridDim.x) * rings;

  // reverse: walk the row pairs from the end - the delta rows the forward kernel wrote LAST are still in L2
  auto phys = [&](long long pair) { return reverse ? n_pairs - 1 - pair : pair; };
  auto issue = [&](int stage, long long pair) {  // producer warp only
    uint8_t* dst = ring + size_t(stage) * stage_bytes;
    const long long r0 = phys(pair) * 2;
    if (r0 + 1 < n_rows) {
      if (lane == 0) {
        ptx::mbar_arrive_expect_tx(&full[stage], static_cast<uint32_t>(stage_bytes));
        ptx::bulk_load_1d(dst, state + r0 * S, static_cast<uint32_t>(state_bytes), &full[stage]);
#pragma unroll
        for (int m = 0; m < NM; ++m)
          ptx::bulk_load_1d(dst + state_bytes + m * delta_bytes, delta + (m * delta_rows + r0) * DP,
                            static_cast<uint32_t>(delta_bytes), &full[stage]);
      }
    } else {  // odd trailing row: 904 bytes is not a bulk-copy size, stage it with plain loads
      float* sd = reinterpret_cast<float*>(dst);
      for (int k = lane; k < S; k += 32) sd[k] = state[r0 * S + k];
#pragma unroll
      for (int m = 0; m < NM; ++m) {
        float* dd = reinterpret_cast<float*>(dst + state_bytes + m * delta_bytes);
        const float* src = delta + (m * delta_rows + r0) * DP;
        for (int k = lane; k < S; k += 32) dd[k] = src[k];
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&full[stage]);
    }
  };

  long long p_issue = t_global;
  if (trank == 0) {
    for (int s = 0; s < stages; ++s, p_issue += t_total)
      if (p_issue < n_pairs) issue(s, p_issue);
  }

  // per-row scalars (active member, step counter) are fetched one pair ahead so their latency never stalls the warp
  auto scalars = [&](long long pair, int& mem, int& stp) {
    const long long row = phys(pair) * 2 + trank;
    mem = 0;
    stp = 0;
    if (pair < n_pairs && row < n_rows) {
      if (member != nullptr) mem = __ldg(member + row);
      if (num_steps != nullptr) stp = num_steps[row];
    }
  };
  int mem_n, stp_n;
  scalars(t_global, mem_n, stp_n);

  int stage = 0;
  uint32_t phase = 0;
  for (long long pair = t_global; pair < n_pairs; pair += t_total) {
    const long long row = phys(pair) * 2 + trank;
    const int mem = mem_n, stp = stp_n;
    scalars(pair + t_total, mem_n, stp_n);
    ptx::mbar_wait(&full[stage], phase);
    if (row < n_rows) {
      uint8_t* base = ring + size_t(stage) * stage_bytes;
      float* s_sm = reinterpret_cast<float*>(base) + trank * S;
      const float* d_sm = reinterpret_cast<const float*>(base + state_bytes) + trank * DP;
      post_tma_row<NM, E, SC>(s_sm, d_sm, 2 * DP, S, row, mem, stp, num_steps != nullptr, next_state, disc, done,
                              num_steps, tc, body, rff, lane);
    }
    // the stage is rewritten by the async proxy next: order this warp's shared-memory accesses before it
    ptx::fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&empty[stage]);
    if (trank == 0) {
      if (p_issue < n_pairs) {
        ptx::mbar_wait(&empty[stage], phase);
        issue(stage, p_issue);
      }
      p_issue += t_total;
    }
    if (++stage == stages) { stage = 0; phase ^= 1; }
  }
}

}  // namespace simstep
