// Grouped, persistent, warp-specialised tcgen05 GEMM for the ensemble MLP layers
// and the random-feature projection:   D[g] = A[g] * B[g]^T  (both K-major).
//
//   * CTA pairs (cta_group::2): two SMs of one TPC own a 256 x 256 output tile.  Each CTA stages its
//     own 128 rows of A and HALF of B (128 of the 256 output features) per k-block, so a pair moves 2 x 32 KB
//     per k-block from L2 where two independent 128 x 256 tiles would move 2 x 48 KB; the leader CTA's single
//     elected thread issues tcgen05.mma.cta_group::2 (M 256, N 256, K 16) reading both CTAs' shared memory,
//     each CTA's TMEM receives its 128 accumulator rows.
//   * A / B tiles arrive by TMA with the 128-byte swizzle through an mbarrier ring; both CTAs'
//     loads complete on the LEADER's full barrier, and the leader's tcgen05.commit multicasts the "stage free"
//     and "accumulator ready" arrivals to both CTAs.
//   * Two 256-column TMEM accumulators are double-buffered so the epilogue of tile i overlaps the MMAs of tile
//     i+1.
//   * The K loop reads the first kb_x blocks from a tensor shared by all groups (the normalised [s,a] input x)
//     and the rest from the group's own activation buffer: that IS the dense-connect concat of
//     BasicMLP.forward (reference milo/milo/dynamics.py:427-430) with no cat kernel.
//   * Epilogues: bias+activation (hidden) or bias+un-normalise (final, dynamics.py:231-232) are written into a
//     swizzled shared-memory staging tile and leave through TMA stores (full 128-byte lines, straight into the
//     next layer's K-slice of the concat buffer); cos/dot for the RFF cost (linear_cost.py:64-71, 96-103)
//     reduces in registers.
#pragma once
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include "ptx.cuh"

namespace simstep {

// depth of the operand ring: 5 x 32 KB + 2 x 16 KB of store staging = 193 KB; 6 fits (225 KB of the 227 KB a CTA
// may use) and was measured, see DESIGN.md section 7
constexpr int kGemmStages = 5;
// staging tiles of the TMA-store epilogue (16 KB each); kOutStages - 1 stores may still be reading shared memory
constexpr int kGemmOutStages = 2;
constexpr int kBlockM = 128;   // accumulator rows per CTA
constexpr int kBlockN = 256;   // accumulator columns (output features per tile)
constexpr int kNumEpiWarps = 4;      // per epilogue group
constexpr int kNumEpiThreads = kNumEpiWarps * 32;
constexpr int kGemmThreads = 64 + kNumEpiThreads;  // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int kTmemCols = 512;                     // two 128x256 fp32 accumulators
constexpr int kABytes = kBlockM * 128;             // one swizzle atom (128 B) per row
constexpr int kOutStageBytes = kBlockM * 128;      // staging tile of the TMA-store epilogue: 128 rows x 128 B
// per-tile epilogue constants staged in shared memory, double-buffered: bias | scale (or cost weights) | shift for
// the tile's kBlockN columns.  Read straight from global memory (one broadcast load per 4 columns per chunk) they
// showed up as the epilogue's dominant stall (long scoreboard on the first use of every chunk).
constexpr int kEpiConstFloats = 3 * kBlockN;
constexpr int kEpiConstBytes = 2 * kEpiConstFloats * 4;

// One ring stage of a CTA: its 128 rows of A and half of the pair's 256 rows of B.
struct GemmShape {
  static constexpr int kBRows = kBlockN / 2;           // B rows staged per CTA
  static constexpr int kBBytes = kBRows * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
};

// Shared-memory plan of one kernel variant.  EG = epilogue warp GROUPS (4 warps each: one per TMEM lane quarter).
// A single epilogue warp per quarter issues about one instruction every five cycles (its chains are dependent), so
// short-K tiles - the first layer, the cost features - are bound by the epilogue, not by the MMAs: with EG = 2 a
// second group takes the upper half of the tile's columns.  Store-tile variants with EG = 2 give every group its own
// pair of staging tiles and pay for them with one ring stage (they are only used where the whole K fits the ring).
template <int EG, bool STORE>
struct GemmPlan {
  static constexpr int kStages = (EG == 2 && STORE) ? 4 : kGemmStages;
  static constexpr int kOutStages = STORE ? kGemmOutStages * EG : 0;
  static constexpr int kThreads = 64 + 128 * EG;  // warp 0 TMA, warp 1 MMA, then the epilogue groups
  static constexpr size_t smem_bytes() {
    return 1024 /*align slack*/ + size_t(kStages) * GemmShape::kStageBytes + size_t(kOutStages) * kOutStageBytes +
           kEpiConstBytes + kBlockM * sizeof(float) /*dot hand-over*/ + 256;
  }
};

// Operand formats.  cvt() is the scalar round-to-operand used by the pack kernels; pack32<RELU>() converts
// 32 fp32 accumulator values (optionally through max(x, 0)) into operand words (32 / 16 of them).
// NaN propagates through every variant (torch.relu(NaN) is NaN); fp16 saturates instead of overflowing.
struct ElemTF32 {
  using storage = float;
  static constexpr int kKind = 0;
  static constexpr uint32_t kFmt = 2;
  static constexpr int kWords32 = 32;  // 32-bit words produced from 32 accumulator values
  __device__ static __forceinline__ storage cvt(float x) { return ptx::round_tf32(x); }
  template <bool RELU>
  __device__ static __forceinline__ void pack32(uint32_t* w, const float (&v)[32]) {
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      float x = v[i];
      if (RELU) asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(x) : "f"(x));
      w[i] = __float_as_uint(ptx::round_tf32(x));
    }
  }
};
struct ElemF16 {
  using storage = __half;
  static constexpr int kKind = 1;
  static constexpr uint32_t kFmt = 0;
  static constexpr int kWords32 = 16;
  __device__ static __forceinline__ storage cvt(float x) {
    uint32_t r;  // saturate instead of overflowing to inf: an exploded state stays finite; NaN stays NaN
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %1;" : "=r"(r) : "f"(x));
    return __ushort_as_half(static_cast<unsigned short>(r & 0xFFFFu));
  }
  template <bool RELU>
  __device__ static __forceinline__ void pack32(uint32_t* w, const float (&v)[32]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      // d = {a -> upper half, b -> lower half}
      if (RELU)
        asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(w[i]) : "f"(v[2 * i + 1]), "f"(v[2 * i]));
      else
        asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(w[i]) : "f"(v[2 * i + 1]), "f"(v[2 * i]));
    }
  }
};
struct ElemBF16 {
  using storage = __nv_bfloat16;
  static constexpr int kKind = 1;
  static constexpr uint32_t kFmt = 1;
  static constexpr int kWords32 = 16;
  __device__ static __forceinline__ storage cvt(float x) { return __float2bfloat16_rn(x); }
  template <bool RELU>
  __device__ static __forceinline__ void pack32(uint32_t* w, const float (&v)[32]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (RELU)
        asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(w[i]) : "f"(v[2 * i + 1]), "f"(v[2 * i]));
      else
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(w[i]) : "f"(v[2 * i + 1]), "f"(v[2 * i]));
    }
  }
};

template <typename E>
struct ElemDims {
  static constexpr int kBlockK = 128 / sizeof(typename E::storage);  // elements per swizzle row
  static constexpr int kUmmaK = 32 / sizeof(typename E::storage);    // K of one tcgen05.mma
};

// kEpiFeat is kEpiRff with the feature-net heads (tanh before the cosine, or no nonlinearity at all) selected at run
// time; it is a separate instantiation so that the random-feature kernel of the env step carries none of that code.
enum EpiMode : int { kEpiHidden = 0, kEpiFinal = 1, kEpiRff = 2, kEpiHiddenTanh = 3, kEpiFeat = 4 };
__host__ __device__ constexpr bool epi_is_rff(int mode) { return mode == kEpiRff || mode == kEpiFeat; }

// Bonus combine of MILO's cost (reference milo/milo/linear_cost.py:96-103, 130-147; GAILCost variants
// gail_cost.py:232-246), applied to one row's feature dot product by the random-feature GEMM's epilogue (the dot
// never leaves registers).
struct CombineArgs {
  int enabled;            // epilogue: finish the row here (needs n_inner == n_tiles)
  const float* disc;      // nullptr: only dot_out is written
  float lambda_b, threshold, c_min, c_max;
  int clamp_cost;
  int transform;          // SIMSTEP_COST_*
  float dot_scale;        // sqrt(2/D), or 1 for a linear head
  float* dot_out;
  float* cost;
  float* ipm;
  float* bonus;
};

__device__ __forceinline__ void combine_row(const CombineArgs& c, long long row, float dot) {
  dot *= c.dot_scale;
  if (c.transform == 1 /*SIMSTEP_COST_GAIL_LS*/) {
    // GAILCost.get_ls_costs (gail_cost.py:232-238): rewards = 1 - 0.25 (1 - d)^2, clipped at 0; cost = -rewards
    const float u = 1.f - dot;
    float r = fmaf(-0.25f * u, u, 1.f);
    if (r < 0.f) r = 0.f;
    dot = -r;
  } else if (c.transform == 2 /*SIMSTEP_COST_GAIL_LL*/) {
    // GAILCost.get_ll_costs (gail_cost.py:240-246): logsigmoid(d) = min(d, 0) - log1p(exp(-|d|))
    dot = fminf(dot, 0.f) - log1pf(expf(-fabsf(dot)));
  }
  if (c.dot_out) c.dot_out[row] = dot;
  if (c.disc == nullptr) return;
  float cc = dot;
  float b;
  if (c.clamp_cost) {
    cc = fminf(fmaxf(cc, c.c_min), c.c_max);
    if (dot != dot) cc = dot;  // torch.clamp keeps NaN
    float dh = c.disc[row] / c.threshold;
    if (dh > 1.0f) dh = 1.0f;
    b = dh * c.c_min;
  } else {
    b = c.disc[row];
  }
  const float i_ = (1.f - c.lambda_b) * cc;
  const float wb = c.lambda_b * b;
  if (c.ipm) c.ipm[row] = i_;
  if (c.bonus) c.bonus[row] = wb;
  if (c.cost) c.cost[row] = i_ - wb;
}

// L2 eviction-priority policies and the hinted forms of the pair's TMA load / the TMA store
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_2d_pair_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int32_t c0,
                                                      int32_t c1, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      :
      : "r"(ptx::smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(bar) & 0xFEFFFFFFu),
        "r"(c0), "r"(c1), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d_hint(const CUtensorMap* map, const void* smem_src, int32_t c0, int32_t c1,
                                                  uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3}], [%1], %4;"
               :
               : "l"(reinterpret_cast<uint64_t>(map)), "r"(ptx::smem_u32(smem_src)), "r"(c0), "r"(c1), "l"(policy)
               : "memory");
}

struct GemmArgs {
  // tile space: tile -> (group, m_tile, n_tile), n fastest; an m_tile is the 256 rows of a CTA pair
  int n_inner;            // consecutive n-tiles of one (group, m_tile) a CTA pair runs back to back (0 / 1: none)
  int group_fastest;      // tile -> (m_tile, group, n_tile): the members of an env tile run side by side on
                          // neighbouring CTA pairs, so the shared x tile is read from HBM once instead of per member
  int reverse;            // walk the tile space backwards: the rows the previous layer wrote LAST (still in L2) first
  int b_evict_last;       // load the weight tiles with the evict_last L2 priority
  int m_tiles;
  int n_tiles;
  int groups;
  // K loop
  int kb_x;               // k-blocks read through tmap_ax (rows shared by all groups)
  int kb_h0;              // first k-block inside tmap_ah
  int kb_h;               // k-blocks read through tmap_ah
  int a_rows_per_group;   // row stride between groups in tmap_ah
  int ax_rows_per_group;  // row stride between groups in tmap_ax (0 when x is shared)
  int b_rows_per_group;
  // epilogue
  const float* bias;      // [groups][n_tiles*kBlockN] or nullptr
  const float* scale;     // kEpiFinal: [n_tiles*kBlockN] or nullptr; kEpiRff: w
  const float* shift;     // kEpiFinal: [n_tiles*kBlockN] or nullptr
  int out_rows_per_group; // hidden / final: row stride between groups in tmap_out
  int out_col0;           // first column (elements) of this layer's output in tmap_out
  void* out;              // kEpiRff: phi float or nullptr
  long long out_pitch;    // kEpiRff: elements
  int rows_valid;         // kEpiRff: rows that exist in `out` and in the combine's outputs
  int cols_valid;
  float rff_phi_scale;    // sqrt(2/D)
  int rff_tanh;           // kEpiRff: phi = cos(tanh(pre-activation)) (MLPCost, linear_cost.py:208-221)
  int rff_linear;         // kEpiRff: phi = pre-activation (discriminator output, gail_cost.py:18-43)
  CombineArgs comb;       // kEpiRff: finish cost / ipm / bonus in the epilogue
};

template <typename E>
__host__ __device__ constexpr uint32_t make_idesc() {
  return (1u << 4)                                        // D format: F32
         | (E::kFmt << 7) | (E::kFmt << 10)               // A / B format
         | (static_cast<uint32_t>(kBlockN >> 3) << 17)    // N
         | (static_cast<uint32_t>((kBlockM * 2) >> 4) << 24);  // M: 256 for a CTA pair
}

// cos(x) for the random-feature epilogue: two-constant Cody-Waite reduction to [-pi, pi] then the SFU
// approximation (abs error < 1e-6 for |x| up to ~1e4, far inside the 1e-3 budget of the cost).
__device__ __forceinline__ float fast_cos(float x) {
  // round-to-nearest through the 1.5 * 2^23 trick (two full-rate FADDs; rintf is an FRND on the quarter-rate pipe
  // that the MUFU.COS below needs too); exact for |x / 2 pi| < 2^22, far beyond any pre-activation seen here
  const float k = (fmaf(x, 0.15915494309189535f, 12582912.f)) - 12582912.f;
  float r = fmaf(k, -6.28318548202514648f, x);   // 2*pi rounded to fp32
  r = fmaf(k, 1.74845553e-7f, r);                // 2*pi_fp32 - 2*pi
  return __cosf(r);
}

// tanh(x) = 1 - 2 / (exp(2x) + 1) on the SFU: absolute error < 5e-7 everywhere (it feeds a cosine, so the absolute
// error is what matters); saturates to +-1 through exp's overflow / underflow.
__device__ __forceinline__ float fast_tanh(float x) {
  const float t = __expf(2.f * x);
  return 1.f - __fdividef(2.f, t + 1.f);
}

template <typename E, int MODE, int EG = 1>
__global__ void __launch_bounds__(64 + 128 * EG, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_ax, const __grid_constant__ CUtensorMap tmap_ah,
                    const __grid_constant__ CUtensorMap tmap_b, const __grid_constant__ CUtensorMap tmap_out,
                    const GemmArgs args) {
  constexpr int CG = 2;  // CTAs per tile
  using S = GemmShape;
  constexpr int BK = ElemDims<E>::kBlockK;
  constexpr int UK = ElemDims<E>::kUmmaK;
  constexpr int kMmasPerBlock = BK / UK;  // 4
  constexpr bool kStoreTile = !epi_is_rff(MODE);
  using Plan = GemmPlan<EG, kStoreTile>;
  constexpr int kStages = Plan::kStages;
  constexpr int kOutStages = Plan::kOutStages;
  constexpr int kEpiWarps = 4 * EG;
  constexpr int kEpiThreads = 128 * EG;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* smem_tiles = smem;                                           // kStages * (A | B)
  uint8_t* smem_out = smem + size_t(kStages) * S::kStageBytes;          // kOutStages staging tiles
  float* smem_const = reinterpret_cast<float*>(smem_out + size_t(kOutStages) * kOutStageBytes);  // [2][kEpiConstFloats]
  float* smem_dot = smem_const + 2 * kEpiConstFloats;  // [kBlockM] second group's partial dots (kEpiRff, EG = 2)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_dot + kBlockM);
  uint64_t* full_bar = bars;                   // [kStages]   (the leader's copy is the one in use)
  uint64_t* empty_bar = bars + kStages;        // [kStages]
  uint64_t* tmem_full_bar = bars + 2 * kStages;      // [2]
  uint64_t* tmem_empty_bar = bars + 2 * kStages + 2; // [2]  (leader's copy)
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = ptx::cluster_ctarank();
  const bool leader = cta_rank == 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full_bar[a], 1);
      ptx::mbar_init(&tmem_empty_bar[a], kEpiWarps * CG);
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tmap_ax);
    ptx::prefetch_tensormap(&tmap_ah);
    ptx::prefetch_tensormap(&tmap_b);
    if (kStoreTile) ptx::prefetch_tensormap(&tmap_out);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_base_smem, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tcgen05_fence_before();
  ptx::cluster_sync();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;
  // everything above overlapped the previous kernel's tail; its outputs are read (and ours written) from here on
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();

  const int total_tiles = args.m_tiles * args.n_tiles * args.groups;
  const int kb_total = args.kb_x + args.kb_h;
  // a CTA pair's iteration `it` runs tile  (tile0 + (it / n_inner) * tile_step) * n_inner + it % n_inner
  const int n_inner = args.n_inner > 1 ? args.n_inner : 1;
  const int total_super = total_tiles / n_inner;
  const int tile0 = blockIdx.x / CG;
  const int tile_step = gridDim.x / CG;
  auto tile_of = [&](int it) {
    int super = tile0 + (it / n_inner) * tile_step;
    if (super >= total_super) return -1;
    if (args.reverse) super = total_super - 1 - super;
    return super * n_inner + it % n_inner;
  };
  auto decode = [&](int tile, int& g, int& m_tile, int& n_tile) {
    n_tile = tile % args.n_tiles;
    const int t2 = tile / args.n_tiles;
    if (args.group_fastest) { g = t2 % args.groups; m_tile = t2 / args.groups; }
    else { m_tile = t2 % args.m_tiles; g = t2 / args.m_tiles; }
  };

  if (warp == 0) {
    // ===== TMA producer (both CTAs of a pair; the leader arms the barrier for both) =====
    // ONE elected thread runs the whole loop (and likewise the MMA issuer below): ptxas then knows the code is
    // single-threaded and emits each TMA / MMA instruction once, instead of wrapping every one of them in an
    // ELECT / BRA.U.ANY loop over the active lanes (about 100 instructions per k-block under `if (lane == 0)`, 40 so)
    if (ptx::elect_one()) {
    const uint64_t pol_last = l2_policy_evict_last();
    int stage = 0;
    uint32_t phase = 0;
    for (int it = 0, tile; (tile = tile_of(it)) >= 0; ++it) {
      int g, m_tile, n_tile;
      decode(tile, g, m_tile, n_tile);
      const int m_row = (m_tile * CG + int(cta_rank)) * kBlockM;
      const int row_ax = g * args.ax_rows_per_group + m_row;
      const int row_ah = g * args.a_rows_per_group + m_row;
      const int row_b = g * args.b_rows_per_group + n_tile * kBlockN + int(cta_rank) * S::kBRows;
      for (int kb = 0; kb < kb_total; ++kb) {
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem_tiles + size_t(stage) * S::kStageBytes;
        uint8_t* sb = sa + kABytes;
        if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], S::kStageBytes * CG);
        if (kb < args.kb_x) {
          ptx::tma_load_2d(sa, &tmap_ax, &full_bar[stage], kb * BK, row_ax);
        } else {
          ptx::tma_load_2d(sa, &tmap_ah, &full_bar[stage], (args.kb_h0 + kb - args.kb_x) * BK, row_ah);
        }
        if (args.b_evict_last) tma_load_2d_pair_hint(sb, &tmap_b, &full_bar[stage], kb * BK, row_b, pol_last);
        else ptx::tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * BK, row_b);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only) =====
    if (leader && ptx::elect_one()) {
      constexpr uint32_t idesc = make_idesc<E>();
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; tile_of(it) >= 0; ++it) {
        const int acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
        ptx::tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kBlockN;
        for (int kb = 0; kb < kb_total; ++kb) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tcgen05_fence_after();
          const uint32_t sa = ptx::smem_u32(smem_tiles + size_t(stage) * S::kStageBytes);
          const uint64_t da = ptx::umma_desc_k_sw128(sa);
          const uint64_t db = ptx::umma_desc_k_sw128(sa + kABytes);
#pragma unroll
          for (int k = 0; k < kMmasPerBlock; ++k) {
            // advance 32 bytes (= UMMA_K elements) along K inside the swizzle atom
            ptx::umma_ss<E::kKind>(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          ptx::umma_commit(&empty_bar[stage]);
          if (kb == kb_total - 1) ptx::umma_commit(&tmem_full_bar[acc]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue warps =====
    const int q = warp & 3;                 // TMEM lane quarter this warp may read
    const int row_in_tile = q * 32 + lane;
    const int epi_tid = threadIdx.x - 64;
    const int grp = epi_tid >> 7;           // epilogue group: owns the columns [grp, grp + 1) * kBlockN / EG of a tile
    const int gtid = epi_tid & 127;
    const uint32_t bar_base = 1 + 3 * grp;  // named barriers of this group (id 3 * EG + 1.. are CTA-wide)
    using T = typename E::storage;
    constexpr bool kFinal = (MODE == kEpiFinal);
    // columns per staging tile (128 bytes per row) and TMEM chunks (32 columns) that fill one
    constexpr int kTileCols = kFinal ? 32 : int(128 / sizeof(T));
    constexpr int kChunksPerStore = kTileCols / 32;
    int store_it = 0;
    float dot = 0.f;  // kEpiRff: feature dot product of this thread's row (carried across a pair's n_inner tiles)
    for (int it = 0, tile; (tile = tile_of(it)) >= 0; ++it) {
      int g, m_tile, n_tile;
      decode(tile, g, m_tile, n_tile);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int n0 = n_tile * kBlockN;
      const int m_row = (m_tile * CG + int(cta_rank)) * kBlockM;
      const float* bias_g = args.bias ? args.bias + size_t(g) * args.n_tiles * kBlockN + n0 : nullptr;
      // stage the tile's per-column constants while the MMAs of this tile are still running: thread t brings
      // columns 2t, 2t + 1 of each vector
      float* cst = smem_const + (it & 1) * kEpiConstFloats;
      if (epi_tid < kBlockN / 2) {
        const int c0 = 2 * epi_tid;
        const float2 bv = bias_g ? __ldg(reinterpret_cast<const float2*>(bias_g + c0)) : make_float2(0.f, 0.f);
        *reinterpret_cast<float2*>(cst + c0) = bv;
        if constexpr (kFinal || epi_is_rff(MODE)) {
          const float fill = kFinal ? 1.f : 0.f;
          const float2 sv = args.scale ? __ldg(reinterpret_cast<const float2*>(args.scale + n0 + c0))
                                       : make_float2(fill, fill);
          *reinterpret_cast<float2*>(cst + kBlockN + c0) = sv;
        }
        if constexpr (kFinal) {
          const float2 hv = args.shift ? __ldg(reinterpret_cast<const float2*>(args.shift + n0 + c0))
                                       : make_float2(0.f, 0.f);
          *reinterpret_cast<float2*>(cst + 2 * kBlockN + c0) = hv;
        }
      }
      ptx::named_bar_sync(3 * EG + 1, kEpiThreads);

      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      ptx::tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kBlockN;
      constexpr int kChunks = kBlockN / 32;
      const int c_begin = grp * (kChunks / EG), c_end = c_begin + kChunks / EG;

      // Two register buffers: the TMEM load of chunk c+1 is in flight while chunk c is processed, and the
      // accumulator is handed back to the MMA warp as soon as the last chunk sits in registers.
      uint32_t ra[32], rb[32];
      ptx::tmem_ld_32x32(taddr + c_begin * 32, ra);

      if (!(args.comb.enabled && it % n_inner != 0)) dot = 0.f;
      auto process = [&](const uint32_t (&r)[32], int c) {
        float v[32];
        {
          const float4* b4 = reinterpret_cast<const float4*>(cst + c * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = b4[j];  // same address in every lane: a shared-memory broadcast
            v[4 * j + 0] = __uint_as_float(r[4 * j + 0]) + b.x;
            v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b.y;
            v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b.z;
            v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b.w;
          }
        }
        if constexpr (kStoreTile) {
          constexpr int kWords = kFinal ? 32 : E::kWords32;  // 32-bit words this chunk contributes to a row
          uint32_t w[kWords];
          if constexpr (kFinal) {
            const float4* s4 = reinterpret_cast<const float4*>(cst + kBlockN + c * 32);
            const float4* h4 = reinterpret_cast<const float4*>(cst + 2 * kBlockN + c * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 sc = s4[j], sh = h4[j];
              v[4 * j + 0] = fmaf(v[4 * j + 0], sc.x, sh.x);
              v[4 * j + 1] = fmaf(v[4 * j + 1], sc.y, sh.y);
              v[4 * j + 2] = fmaf(v[4 * j + 2], sc.z, sh.z);
              v[4 * j + 3] = fmaf(v[4 * j + 3], sc.w, sh.w);
            }
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = __float_as_uint(v[j]);
          } else if constexpr (MODE == kEpiHiddenTanh) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = tanhf(v[j]);
            E::template pack32<false>(w, v);
          } else {
            E::template pack32<true>(w, v);
          }
          // staging tile: row r holds 128 bytes, 16-byte unit j sits at unit j ^ (r & 7) (TMA SWIZZLE_128B)
          const int sub = c % kChunksPerStore;            // position of this chunk inside the staging row
          constexpr int kGroupStages = kGemmOutStages;  // staging tiles owned by one group
          const int buf = grp * kGroupStages + store_it % kGroupStages;
          if (sub == 0) {
            // the TMA store that last read this staging buffer must have finished reading shared memory
            if (gtid == 0) ptx::tma_store_wait_read<kGroupStages - 1>();
            ptx::named_bar_sync(bar_base, 128);
          }
          uint8_t* srow = smem_out + size_t(buf) * kOutStageBytes + row_in_tile * 128;
          constexpr int kUnits = kWords / 4;              // 16-byte units written per chunk
#pragma unroll
          for (int u = 0; u < kUnits; ++u) {
            const int unit = sub * kUnits + u;
            *reinterpret_cast<uint4*>(srow + ((unit ^ (row_in_tile & 7)) << 4)) =
                make_uint4(w[4 * u], w[4 * u + 1], w[4 * u + 2], w[4 * u + 3]);
          }
          if (sub == kChunksPerStore - 1) {
            ptx::fence_proxy_async_smem();
            ptx::named_bar_sync(bar_base + 1, 128);
            if (gtid == 0) {
              const int col = args.out_col0 + n0 + (c / kChunksPerStore) * kTileCols;
              ptx::tma_store_2d(&tmap_out, smem_out + size_t(buf) * kOutStageBytes, col,
                                g * args.out_rows_per_group + m_row);
              ptx::tma_store_commit();
            }
            ++store_it;
          }
        } else {  // kEpiRff: phi = cos(pre-activation); dot with w (padded columns carry w == 0)
          const long long row = static_cast<long long>(m_row) + row_in_tile;
          const float4* w4 = reinterpret_cast<const float4*>(cst + kBlockN + c * 32);
          float f[32];
          if constexpr (MODE == kEpiFeat) {
            if (args.rff_linear) {
#pragma unroll
              for (int j = 0; j < 32; ++j) f[j] = v[j];
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) f[j] = __cosf(fast_tanh(v[j]));  // |tanh| <= 1: no range reduction needed
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) f[j] = fast_cos(v[j]);
          }
          if (args.scale != nullptr) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 w = w4[j];
              dot = fmaf(f[4 * j + 0], w.x, dot);
              dot = fmaf(f[4 * j + 1], w.y, dot);
              dot = fmaf(f[4 * j + 2], w.z, dot);
              dot = fmaf(f[4 * j + 3], w.w, dot);
            }
          }
          if (args.out != nullptr && row < args.rows_valid) {
            float* prow = static_cast<float*>(args.out) + row * args.out_pitch + n0 + c * 32;
            const int col = n0 + c * 32;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col + j < args.cols_valid) prow[j] = f[j] * args.rff_phi_scale;
          }
        }
      };

#pragma unroll 1
      for (int c = c_begin; c < c_end; c += 2) {
        ptx::tmem_ld_wait();
        ptx::tmem_ld_32x32(taddr + (c + 1) * 32, rb);
        process(ra, c);
        ptx::tmem_ld_wait();
        if (c + 2 < c_end) {
          ptx::tmem_ld_32x32(taddr + (c + 2) * 32, ra);
        } else {
          // accumulator drained: the MMA warp (leader CTA) may overwrite it
          ptx::tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
        }
        process(rb, c + 1);
      }
      if constexpr (epi_is_rff(MODE)) {
        const long long row = static_cast<long long>(m_row) + row_in_tile;
        const bool finish = !args.comb.enabled || it % n_inner == n_inner - 1;  // the row's dot leaves registers
        float total = dot;
        if constexpr (EG == 2) {
          if (finish && args.scale != nullptr) {  // the upper group hands its part of the dot product over
            if (grp == 1) smem_dot[row_in_tile] = dot;
            ptx::named_bar_sync(3 * EG + 2, kEpiThreads);
            total = dot + smem_dot[row_in_tile];
            // the next hand-over is behind the next tile's constants barrier, which every group-0 thread passes
            // only after this read
          }
        }
        if (grp == 0 && finish && args.comb.enabled && row < args.rows_valid) combine_row(args.comb, row, total);
      }
    }
    if (kStoreTile && gtid == 0) ptx::tma_store_wait<0>();  // shared memory must outlive the last store's read
  }

  ptx::tcgen05_fence_before();
  ptx::cluster_sync();  // nobody leaves while its peer can still signal it
  if (warp == 1) {
    ptx::tcgen05_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace simstep
