// The whole ensemble forward pass (reference milo/milo/dynamics.py:422-433, BasicMLP.forward of every member, and the
// un-normalisation of dynamics.py:231-232) as ONE persistent launch whose work unit is a COLUMN of the layer stack:
//
//     unit = (env tile of 256 rows, member);   a CTA pair runs  layer 1 (n-tiles 0, 1) -> layer 2 -> ... -> final
//
// for its unit and then takes the next unit.  Dense-connect makes layer l+1 of a (member, env tile) depend on layer l
// of the SAME (member, env tile) only, and with cta_group::2 each CTA of the pair both loads (A operand) and stores
// (epilogue) its own 128 rows - so the dependency never leaves the CTA:
//
//   * the epilogue publishes "hidden tile k of this CTA has been stored" through a shared-memory counter after the
//     tile's TMA stores have COMPLETED (cp.async.bulk.wait_group, not .read); the TMA producer looks at the counter
//     only before the first k-block that comes from that tile's 256 columns.  No global-memory flags, no gpu-scope
//     fences, no other CTA is waited for (the per-layer tile order of the earlier fused experiment needed both).
//   * the K loop of layer l+1 reads [x | h_1 | ... | h_l] in that order, so the blocks that depend on the tile just
//     finished come LAST: the MMAs of the next layer start on x and the older slices while the epilogue drains.
//   * the activation rows of a unit are written and read back by the same SM pair within tens of microseconds, i.e.
//     they are L2 hits: the final layer (HBM-bound when launched alone: it re-reads a member's whole 4.6 KB concat
//     row for 226 outputs) and the short first layer (epilogue-bound alone) disappear into the tensor-bound average.
//   * ACTIVATION SLOTS: a pair keeps a whole unit's activation rows in ITS OWN 256-row slot of the activation buffer
//     instead of at the unit's rows - the live part of the buffer is then 74 pairs x 256 rows x 4 KB = 78 MB whatever
//     the batch.  Safe without extra synchronisation: the first store into the slot for unit u+1 follows an MMA that
//     was issued after every MMA of unit u, and those had consumed every load from the slot.  (The shared units of the
//     last round, below, keep their rows at the unit's env rows, where both pairs find them.)
//   * THE LAST, PARTIAL ROUND.  628 units of the bench batch are 8 rounds of 74 pairs plus 36 units; run as a ninth
//     round they leave 38 pairs idle for a whole unit (6 % of the launch).  When the T left-over units are at most half
//     the pairs, TWO pairs share each of them: pair 2u + p computes the n-tiles n % 2 == p of every hidden layer and the
//     column half p of every final-layer tile (an M 256 x N 128 product), so the last round takes half a unit.  Only
//     here does a dependency cross CTA pairs: the epilogue also publishes its tile count in global memory
//     (st.release.gpu) and the partner's producer polls it (ld.acquire.gpu) before the k-blocks that come from the
//     partner's column tiles; the reader zeroes the counter when it is through, so the buffer is clean for the next
//     launch (and for CUDA-graph replays).  All pairs are co-resident (one CTA per SM), nobody waits on work that has
//     not been scheduled.
//
//   * ORDER OF THE UNITS.  Whole rounds take the members of an env tile in sequence on one pair (all pairs then stream
//     the same member's weights at any time: 1.5 % faster than members side by side); the units that do not fill a
//     whole number of such rounds go round-robin, and the last partial round is shared as described above.
//   * L2 PRIORITIES.  Weights and activations are loaded and stored evict_last: every unit of a member re-reads the
//     same weights, a unit re-reads its own rows layer after layer (measured 2.5 % faster on the launch, and 2.5 us
//     slower on the post-step kernel, whose delta rows find less room in L2; marking x and the output evict_first on
//     top was measured neutral).
//
// Tried and dropped: a cluster of FOUR CTAs per unit (both pairs on one unit throughout, the A operand multicast between
// them: 25 % fewer bytes out of L2, bit-identical results).  Only 33 such clusters are co-schedulable on the 148 SMs
// (GPC sizes), 132 SMs instead of 148, and the launch was 12 % slower; the multicast itself changed nothing.  Also
// tried: running the first layer of the NEXT unit in front of the final layer of the current one (two slots per pair),
// so that the short first layer's epilogues drain behind 36 k-blocks of MMAs - bit-identical, 1 % slower.  And the env
// step's tail (next state, discrepancy, termination) on four extra warps of this kernel, for the env tiles whose
// members had all run on one pair: correct, and break-even, because this kernel is bound by the L2 -> SM path that the
// tail's bytes need as well (DESIGN.md section 5).
//
// Pipeline, barriers, TMEM double-buffering, the operand ring and the TMA-store epilogue are those of
// gemm_tcgen05.cuh (one epilogue group); the accumulation order of every output element is the same as in
// the per-layer launches, so the results are bit-identical to them.
#pragma once
#include <type_traits>
#include "gemm_tcgen05.cuh"

#ifndef SIMSTEP_MAX_HIDDEN
#define SIMSTEP_MAX_HIDDEN 8
#endif

namespace simstep {

constexpr int kChainMaxLayers = SIMSTEP_MAX_HIDDEN + 1;

struct ChainLayer {
  int n_tiles;            // n-tiles (256 output columns each) per unit
  int kb_x, kb_h0, kb_h;  // K loop: k-blocks from x, first k-block / number of k-blocks from the activation buffer
  int b_rows_per_group;   // packed weight rows per member
  int out_col0;           // hidden layers: first column of the output slice in the activation buffer
  const float* bias;      // [groups][n_tiles * kBlockN] or nullptr
};

constexpr int kChainMaxDepTiles = 64;

struct ChainArgs {
  int n_layers;            // hidden layers + the final one (the last entry of layer[])
  int m_tiles, groups;
  int a_rows_per_group;    // row stride between members in the activation buffer (shared units; whole units use slots)
  int out_rows_per_group;  // row stride between members in the final output (delta workspace)
  int hidden_tiles;        // hidden tiles per unit (sum of n_tiles over the hidden layers)
  const float* scale;      // final layer: [n_tiles * kBlockN] or nullptr (dynamics.py:231-232)
  const float* shift;
  // the last, partial round: units [units - tail_units, units) are shared by two pairs each (0: plain extra round)
  int tail_units;
  int seq_rounds;          // whole rounds run with the members of an env tile in sequence on one pair (0: none)
  int tiles_per_role[2];                      // hidden tiles role p stores per shared unit
  unsigned char dep_role[kChainMaxDepTiles];  // column tile T of the activation buffer: the role that stores it ...
  unsigned char dep_ord[kChainMaxDepTiles];   // ... and its ordinal among that role's tiles of the unit
  unsigned int* tail_cnt;                     // [tail_units][2 roles][2 row halves], zero between launches
  ChainLayer layer[kChainMaxLayers];
};

struct ChainMaps {
  CUtensorMap x, h, out_final;
  CUtensorMap w[kChainMaxLayers];
  CUtensorMap w_final64;   // the final layer's weights with a 64-row box (column halves of the shared units)
};

__device__ __forceinline__ uint32_t ld_acquire_cta_smem(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(ptx::smem_u32(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_cta_smem(uint32_t* p, uint32_t v) {
  asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(ptx::smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void chain_fence_proxy_async_global() {
  asm volatile("fence.proxy.async.global;" ::: "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const unsigned int* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned int* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
template <typename E>
__host__ __device__ constexpr uint32_t make_idesc_n(int n) {
  return (1u << 4) | (E::kFmt << 7) | (E::kFmt << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>((kBlockM * 2) >> 4) << 24);
}

// One work item of a CTA pair: a whole unit (role < 0) or one of the two roles of a shared unit of the last round.
struct ChainItem {
  int unit;
  int role;
};
// Host side of the schedule: how many CTA pairs run, how many whole rounds take an env tile's members in sequence, and how
// many units of the last partial round are shared between two pairs (0: it runs as a plain round).  Used by the launcher
// and by simstep_debug_chain_schedule (the CPU test of this arithmetic).
inline void chain_schedule(int m_tiles, int groups, int max_pairs, bool share, int* pairs, int* seq_rounds,
                           int* tail_units) {
  const int units = m_tiles * groups;
  *pairs = units < max_pairs ? units : max_pairs;
  if (*pairs < 1) *pairs = 1;
  *seq_rounds = units > *pairs ? m_tiles / *pairs : 0;
  const int tail = (units - *seq_rounds * *pairs * groups) % *pairs;
  *tail_units = (share && tail > 0 && 2 * tail <= *pairs) ? tail : 0;
}

__host__ __device__ __forceinline__ bool chain_item(const ChainArgs& a, int pair, int pairs, int i, ChainItem& it) {
  // seq_rounds whole rounds in which a pair takes ALL members of an env tile one after the other (the members of an env
  // tile then meet inside one CTA pair) ...
  const int seq_items = a.seq_rounds * a.groups;
  if (i < seq_items) {
    it.unit = (pair + (i / a.groups) * pairs) * a.groups + i % a.groups;
    it.role = -1;
    return true;
  }
  // ... then the remaining units round-robin, the last partial round shared between pairs
  const int units = a.m_tiles * a.groups;
  const int base = a.seq_rounds * pairs * a.groups;
  const int full_units = units - a.tail_units;
  const int j = i - seq_items;
  const int u = base + pair + j * pairs;
  if (u < full_units) { it.unit = u; it.role = -1; return true; }
  const int n_full = full_units > base + pair ? (full_units - base - pair + pairs - 1) / pairs : 0;
  if (j == n_full && pair < 2 * a.tail_units) { it.unit = full_units + (pair >> 1); it.role = pair & 1; return true; }
  return false;
}

template <typename E, bool TANH>
__global__ void __launch_bounds__(kGemmThreads, 1)
ensemble_chain_kernel(const __grid_constant__ ChainMaps maps, const __grid_constant__ ChainArgs args) {
  constexpr int CG = 2;
  using S = GemmShape;
  using Plan = GemmPlan<1, true>;
  constexpr int BK = ElemDims<E>::kBlockK;
  constexpr int UK = ElemDims<E>::kUmmaK;
  constexpr int kMmasPerBlock = BK / UK;
  constexpr int kStages = Plan::kStages;
  constexpr int kOutStages = Plan::kOutStages;
  constexpr int kKbPerTile = kBlockN / BK;  // k-blocks of the activation buffer that one hidden tile produces
  constexpr int kHalfN = kBlockN / 2;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* smem_tiles = smem;
  uint8_t* smem_out = smem + size_t(kStages) * S::kStageBytes;
  float* smem_const = reinterpret_cast<float*>(smem_out + size_t(kOutStages) * kOutStageBytes);
  float* smem_dot = smem_const + 2 * kEpiConstFloats;  // unused here; keeps GemmPlan's layout
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_dot + kBlockM);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tmem_full_bar = bars + 2 * kStages;
  uint64_t* tmem_empty_bar = bars + 2 * kStages + 2;
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);
  uint32_t* stored_cnt = tmem_base_smem + 1;  // hidden tiles of THIS CTA whose stores have completed

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
      ptx::mbar_init(&tmem_empty_bar[a], kNumEpiWarps * CG);
    }
    *stored_cnt = 0;
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&maps.x);
    ptx::prefetch_tensormap(&maps.h);
    ptx::prefetch_tensormap(&maps.out_final);
    for (int l = 0; l < args.n_layers; ++l) ptx::prefetch_tensormap(&maps.w[l]);
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_base_smem, kTmemCols);
    ptx::tmem_relinquish();
  }
  ptx::tcgen05_fence_before();
  ptx::cluster_sync();
  ptx::tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;
  ptx::grid_dep_wait();
  ptx::grid_dep_launch();

  const int pair = blockIdx.x / CG;
  const int pairs = gridDim.x / CG;
  const int n_hidden = args.n_layers - 1;
  const int slot_row = (pair * CG + int(cta_rank)) * kBlockM;
  // Tiles of layer l an item runs: every n-tile of a whole unit; of a shared unit the n-tiles n % 2 == role of a hidden
  // layer and the column half `role` of every final-layer tile.
  auto n_begin = [&](const ChainItem& it, int l) { return (it.role < 0 || l == n_hidden) ? 0 : it.role; };
  auto n_step = [&](const ChainItem& it, int l) { return (it.role < 0 || l == n_hidden) ? 1 : 2; };

  if (warp == 0) {
    // ===== TMA producer (both CTAs; the leader arms the barrier for both) =====
    // ONE elected thread runs the whole loop: ptxas then knows the code is single-threaded and emits each TMA / MMA
    // instruction once, instead of wrapping every one of them in an ELECT / BRA.U.ANY loop over the active lanes
    // (about 100 instructions per k-block when the issue sits under `if (lane == 0)`, 40 this way)
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint64_t pol_last = l2_policy_evict_last();
      uint32_t have = 0;       // last value seen in stored_cnt
      uint32_t done_tiles = 0; // hidden tiles this CTA stored in the items before the current one
      ChainItem item;
      for (int i = 0; chain_item(args, pair, pairs, i, item); ++i) {
        const bool shared = item.role >= 0;
        const int g = item.unit % args.groups;
        const int m_row = ((item.unit / args.groups) * CG + int(cta_rank)) * kBlockM;
        const int row_ah = shared ? g * args.a_rows_per_group + m_row : slot_row;
        // shared unit: the partner's tile counter for this row half (polled), zeroed again when this item is through
        unsigned int* partner_cnt = nullptr;
        uint32_t have_partner = 0;
        if (shared)
          partner_cnt = args.tail_cnt + (((item.unit - (args.m_tiles * args.groups - args.tail_units)) * 2 +
                                          (1 - item.role)) * 2 + int(cta_rank));
        for (int l = 0; l < args.n_layers; ++l) {
          const ChainLayer& ly = args.layer[l];
          const bool half = shared && l == n_hidden;
          const int kb_total = ly.kb_x + ly.kb_h;
          const uint32_t stage_bytes = uint32_t(kABytes + (half ? S::kBBytes / 2 : S::kBBytes)) * CG;
          const CUtensorMap* wmap = half ? &maps.w_final64 : &maps.w[l];
          for (int n_tile = n_begin(item, l); n_tile < ly.n_tiles; n_tile += n_step(item, l)) {
            // weight rows of this CTA: half of the pair's 256 (or, for a column half, 128) output features
            const int row_b = g * ly.b_rows_per_group + n_tile * kBlockN +
                              (half ? item.role * kHalfN + int(cta_rank) * (kHalfN / 2) : int(cta_rank) * S::kBRows);
            for (int kb = 0; kb < kb_total; ++kb) {
              const int hk = ly.kb_h0 + kb - ly.kb_x;  // k-block inside the activation buffer (kb >= kb_x)
              if (kb >= ly.kb_x) {
                const int t = hk / kKbPerTile;         // column tile of the activation buffer
                if (!shared || args.dep_role[t] == item.role) {
                  const uint32_t need = done_tiles + (shared ? uint32_t(args.dep_ord[t]) : uint32_t(t)) + 1u;
                  if (have < need) {
                    unsigned int spins = 0;
                    while ((have = ld_acquire_cta_smem(stored_cnt)) < need) {
                      __nanosleep(32);
                      if (++spins > (1u << 26)) __trap();  // a dependency that never arrives is a bug: trap, do not hang
                    }
                    chain_fence_proxy_async_global();  // the rows are read by the async proxy (TMA) next
                  }
                } else {
                  const uint32_t need = uint32_t(args.dep_ord[t]) + 1u;
                  if (have_partner < need) {
                    unsigned int spins = 0;
                    while ((have_partner = ld_acquire_gpu_u32(partner_cnt)) < need) {
                      __nanosleep(64);
                      // the partner pair may not even be resident yet when other kernels share the GPU: ~20 s of patience
                      if (++spins > (1u << 28)) __trap();
                    }
                    chain_fence_proxy_async_global();
                  }
                }
              }
              ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
              uint8_t* sa = smem_tiles + size_t(stage) * S::kStageBytes;
              uint8_t* sb = sa + kABytes;
              if (leader) ptx::mbar_arrive_expect_tx(&full_bar[stage], stage_bytes);
              if (kb < ly.kb_x) ptx::tma_load_2d(sa, &maps.x, &full_bar[stage], kb * BK, m_row);
              else tma_load_2d_pair_hint(sa, &maps.h, &full_bar[stage], hk * BK, row_ah, pol_last);
              tma_load_2d_pair_hint(sb, wmap, &full_bar[stage], kb * BK, row_b, pol_last);
              if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
          }
        }
        if (shared) {
          // every tile the partner stores has been seen (the final layer reads them all): leave the counter clean
          if (args.tiles_per_role[1 - item.role] > 0) *partner_cnt = 0u;
          done_tiles += uint32_t(args.tiles_per_role[item.role]);
        } else {
          done_tiles += uint32_t(args.hidden_tiles);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only) =====
    if (leader && ptx::elect_one()) {
      constexpr uint32_t idesc_full = make_idesc_n<E>(kBlockN);
      constexpr uint32_t idesc_half = make_idesc_n<E>(kHalfN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      ChainItem item;
      for (int i = 0; chain_item(args, pair, pairs, i, item); ++i) {
        for (int l = 0; l < args.n_layers; ++l) {
          const int kb_total = args.layer[l].kb_x + args.layer[l].kb_h;
          const uint32_t idesc = (item.role >= 0 && l == n_hidden) ? idesc_half : idesc_full;
          for (int n_tile = n_begin(item, l); n_tile < args.layer[l].n_tiles; n_tile += n_step(item, l), ++it) {
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
              for (int k = 0; k < kMmasPerBlock; ++k)
                ptx::umma_ss<E::kKind>(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
              ptx::umma_commit(&empty_bar[stage]);
              if (kb == kb_total - 1) ptx::umma_commit(&tmem_full_bar[acc]);
              if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue warps =====
    const int q = warp & 3;
    const int row_in_tile = q * 32 + lane;
    const int epi_tid = threadIdx.x - 64;
    using T = typename E::storage;
    int store_it = 0;
    int it = 0;
    uint32_t published = 0;   // epi_tid 0: value last written to stored_cnt
    bool pending = false;     // epi_tid 0: the previous hidden tile's stores are committed but not yet published
    ChainItem item;
    for (int i = 0; chain_item(args, pair, pairs, i, item); ++i) {
      const bool shared = item.role >= 0;
      const int g = item.unit % args.groups;
      const int m_row = ((item.unit / args.groups) * CG + int(cta_rank)) * kBlockM;
      const int row_h = shared ? g * args.a_rows_per_group + m_row : slot_row;
      unsigned int* my_cnt = nullptr;   // shared unit: this CTA's tile counter, read by the partner pair
      uint32_t my_tiles = 0;
      if (shared)
        my_cnt = args.tail_cnt + (((item.unit - (args.m_tiles * args.groups - args.tail_units)) * 2 + item.role) * 2 +
                                  int(cta_rank));
      for (int l = 0; l < args.n_layers; ++l) {
        const ChainLayer& ly = args.layer[l];
        const bool is_final = l == n_hidden;
        const bool half = shared && is_final;
        for (int n_tile = n_begin(item, l); n_tile < ly.n_tiles; n_tile += n_step(item, l), ++it) {
          const int acc = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          const int n0 = n_tile * kBlockN + (half ? item.role * kHalfN : 0);
          const float* bias_g = ly.bias ? ly.bias + size_t(g) * ly.n_tiles * kBlockN + n0 : nullptr;
          // stage the tile's per-column constants while its MMAs are still running
          float* cst = smem_const + (it & 1) * kEpiConstFloats;
          if (!half || epi_tid < kHalfN / 2) {
            const int c0 = 2 * epi_tid;
            const float2 bv = bias_g ? __ldg(reinterpret_cast<const float2*>(bias_g + c0)) : make_float2(0.f, 0.f);
            *reinterpret_cast<float2*>(cst + c0) = bv;
            if (is_final) {
              const float2 sv = args.scale ? __ldg(reinterpret_cast<const float2*>(args.scale + n0 + c0))
                                           : make_float2(1.f, 1.f);
              const float2 hv = args.shift ? __ldg(reinterpret_cast<const float2*>(args.shift + n0 + c0))
                                           : make_float2(0.f, 0.f);
              *reinterpret_cast<float2*>(cst + kBlockN + c0) = sv;
              *reinterpret_cast<float2*>(cst + 2 * kBlockN + c0) = hv;
            }
          }
          ptx::named_bar_sync(4, kNumEpiThreads);

          ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
          ptx::tcgen05_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * kBlockN;
          uint32_t ra[32], rb[32];
          ptx::tmem_ld_32x32(taddr, ra);

          // one 32-column chunk of this thread's row: bias (+ scale/shift | activation + convert) into the swizzled
          // staging tile; a full staging tile (128 rows x 128 bytes) leaves through one TMA store
          auto process = [&](auto final_tag, const uint32_t (&r)[32], int c) {
            constexpr bool kFinal = decltype(final_tag)::value;
            constexpr int kTileCols = kFinal ? 32 : int(128 / sizeof(T));
            constexpr int kChunksPerStore = kTileCols / 32;
            constexpr int kWords = kFinal ? 32 : E::kWords32;
            float v[32];
            {
              const float4* b4 = reinterpret_cast<const float4*>(cst + c * 32);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 b = b4[j];
                v[4 * j + 0] = __uint_as_float(r[4 * j + 0]) + b.x;
                v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + b.y;
                v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + b.z;
                v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + b.w;
              }
            }
            uint32_t w[kWords];
            if constexpr (kFinal) {
              const float4* s4 = reinterpret_cast<const float4*>(cst + kBlockN + c * 32);
              const float4* h4 = reinterpret_cast<const float4*>(cst + 2 * kBlockN + c * 32);
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float4 sc = s4[j], sh = h4[j];
                w[4 * j + 0] = __float_as_uint(fmaf(v[4 * j + 0], sc.x, sh.x));
                w[4 * j + 1] = __float_as_uint(fmaf(v[4 * j + 1], sc.y, sh.y));
                w[4 * j + 2] = __float_as_uint(fmaf(v[4 * j + 2], sc.z, sh.z));
                w[4 * j + 3] = __float_as_uint(fmaf(v[4 * j + 3], sc.w, sh.w));
              }
            } else if constexpr (TANH) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = tanhf(v[j]);
              E::template pack32<false>(w, v);
            } else {
              E::template pack32<true>(w, v);
            }
            const int sub = c % kChunksPerStore;
            const int buf = store_it % kOutStages;
            if (sub == 0) {
              if (epi_tid == 0) ptx::tma_store_wait_read<kOutStages - 1>();
              ptx::named_bar_sync(1, kNumEpiThreads);
            }
            uint8_t* srow = smem_out + size_t(buf) * kOutStageBytes + row_in_tile * 128;
            constexpr int kUnits = kWords / 4;
#pragma unroll
            for (int u = 0; u < kUnits; ++u) {
              const int unit16 = sub * kUnits + u;
              *reinterpret_cast<uint4*>(srow + ((unit16 ^ (row_in_tile & 7)) << 4)) =
                  make_uint4(w[4 * u], w[4 * u + 1], w[4 * u + 2], w[4 * u + 3]);
            }
            if (sub == kChunksPerStore - 1) {
              ptx::fence_proxy_async_smem();
              ptx::named_bar_sync(2, kNumEpiThreads);
              if (epi_tid == 0) {
                const int col = (kFinal ? 0 : ly.out_col0) + n0 + (c / kChunksPerStore) * kTileCols;
                if constexpr (kFinal)
                  ptx::tma_store_2d(&maps.out_final, smem_out + size_t(buf) * kOutStageBytes, col,
                                    g * args.out_rows_per_group + m_row);
                else
                  tma_store_2d_hint(&maps.h, smem_out + size_t(buf) * kOutStageBytes, col, row_h, l2_policy_evict_last());
                ptx::tma_store_commit();
                if (pending) {
                  // the previous hidden tile (same layer: nothing this CTA runs next reads it yet) - every group but
                  // the one just committed has completed by now, the wait returns at once
                  ptx::tma_store_wait<1>();
                  chain_fence_proxy_async_global();
                  st_release_cta_smem(stored_cnt, ++published);
                  pending = false;
                }
              }
              ++store_it;
            }
          };
          auto run_tile = [&](auto final_tag, int n_chunks) {
#pragma unroll 1
            for (int c = 0; c < n_chunks; c += 2) {
              ptx::tmem_ld_wait();
              ptx::tmem_ld_32x32(taddr + (c + 1) * 32, rb);
              process(final_tag, ra, c);
              ptx::tmem_ld_wait();
              if (c + 2 < n_chunks) {
                ptx::tmem_ld_32x32(taddr + (c + 2) * 32, ra);
              } else {
                ptx::tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
              }
              process(final_tag, rb, c + 1);
            }
          };
          if (is_final) {
            run_tile(std::true_type{}, (half ? kHalfN : kBlockN) / 32);
          } else {
            run_tile(std::false_type{}, kBlockN / 32);
            if (epi_tid == 0) {
              if (!shared && n_tile + 1 < ly.n_tiles) {
                pending = true;   // the next tile (same layer) does not read this one: publish behind its first store
              } else {
                // the next layer's K loop ends in these columns: publish as soon as the stores have landed
                ptx::tma_store_wait<0>();
                chain_fence_proxy_async_global();
                published += pending ? 2u : 1u;
                pending = false;
                st_release_cta_smem(stored_cnt, published);
                if (shared) st_release_gpu_u32(my_cnt, ++my_tiles);  // ... and the partner pair's next layer too
              }
            }
          }
        }
      }
    }
    if (epi_tid == 0) ptx::tma_store_wait<0>();
  }

  ptx::tcgen05_fence_before();
  ptx::cluster_sync();
  if (warp == 1) {
    ptx::tcgen05_fence_after();
    ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

}  // namespace simstep
