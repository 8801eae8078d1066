// C ABI of libsimstep.so (see include/simstep.h): handle, operand packing,
// workspaces, tensor maps and the launch sequences of the env step.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/simstep.h"
#include "elementwise.cuh"
#include "gemm_tcgen05.cuh"
#include "final_launch.h"
#include "chain_launch.h"
#include "imitation.cuh"
#include "imitation_h3d.cuh"
#include "npg.cuh"
#include "policy.cuh"
#include "post_tma.cuh"
#include "train.cuh"

using namespace simstep;

namespace {

std::atomic<long long> g_launches{0};
thread_local std::string g_create_error;

inline long long round_up(long long x, long long m) { return (x + m - 1) / m * m; }

constexpr int kMaxDevices = 64;  // per-device bookkeeping of kernel attributes / scratch buffers

struct Layer {
  int in_ref = 0;   // reference nn.Linear in_features
  int out = 0;      // out_features
  int o_pad = 0;    // rows of the packed operand (multiple of kBlockN)
  int k_pad = 0;    // packed K (multiple of the swizzle row)
  int kb_x = 0, kb_h0 = 0, kb_h = 0;
  int out_col0 = 0; // column of this layer's output inside the activation buffer
  PackSegs segs{};
  void* w = nullptr;      // [N][o_pad][k_pad] operand storage
  float* bias = nullptr;  // [N][o_pad]
  CUtensorMap tmap_w;
  CUtensorMap tmap_w64;  // the same operand with a 64-row box (column halves of the chain kernel's shared units)
};

}  // namespace

struct simstep_handle {
  simstep_config cfg{};
  int device = 0;
  int sm_count = 148;
  int esize = 4;  // bytes per GEMM operand element
  int bk = 32;    // elements per 128-byte swizzle row
  int cg = 2;     // CTAs per GEMM tile: 2 = cta_group::2 pairs (256-row tiles), 1 = single-CTA tiles
  int row_align = 256;  // workspace rows are padded to whole tiles
  int S = 0, A = 0, N = 0, L = 0;
  int XP = 0, HT = 0, SP = 0;
  int DP = 0;  // pitch (floats) of the fp32 delta workspace rows: S rounded up to 4, so a row is 16-byte granular
  std::vector<Layer> layers;  // L hidden + 1 final
  unsigned long long* sat_dev = nullptr;  // normalised inputs beyond the fp16 range seen so far (prep kernel)
  float* tf_dev = nullptr;         // mean_s | scale_s | mean_a | scale_a
  float* out_scale_dev = nullptr;  // [SP]
  float* out_shift_dev = nullptr;  // [SP]
  bool have_ensemble = false;

  long long cap_rows = 0;
  void* xbuf = nullptr;
  void* hbuf = nullptr;
  float* dws = nullptr;
  unsigned int* tickets = nullptr;  // fused final layer: one arrival counter per 128-row block (gemm_final.cuh)
  // SIMSTEP_DEBUG_GUARDS=1 (read at simstep_create): every workspace buffer sits between two 64 KB guard zones filled with
  // 0xA5; simstep_debug_check_guards counts the guard bytes that no longer are (compute-sanitizer is not available on
  // the GPU boxes: this is the out-of-bounds check the test suite runs instead)
  bool guards_on = false;
  std::vector<std::pair<void*, size_t>> guard_allocs;  // (user pointer, user bytes)
  long long tail_rows_done = 0;       // rows [0, tail_rows_done) of the chunk had their step tail run inside the chain kernel
  bool forward_was_chain = false;     // the workspace's deltas were written by the chain kernel (in row order)
  unsigned int* chain_cnt = nullptr;  // chain kernel: tile counters of the shared units of the last round (zero between launches)
  CUtensorMap tmap_x, tmap_h, tmap_dws;

  // RFF cost
  bool have_rff = false;
  int D = 0, D_pad = 0, rff_in = 0, RK = 0, RKT = 0;
  int rff_split_cap = 0;  // operands were packed as hi/lo pairs: rows hold [hi | lo], weights [hi | hi | lo]
  int rff_split = 0;      // the three-product evaluation is in use (simstep_set_rff_split; needs rff_split_cap)
  int rff_col2 = 0;  // input_type 'ss': operand column of s' (s sits at 0); the weight columns are packed to match
  void* rff_w = nullptr;
  float* rff_b = nullptr;
  float* rff_wpad = nullptr;
  void* rffin = nullptr;
  float* rff_part = nullptr;
  double* colsum_partial = nullptr;
  CUtensorMap tmap_rffw, tmap_rffin;
  // feature net (MLPCost): hidden layers of this handle feed the cos-feature head instead of a packed input row
  bool feat_net = false;
  int feat_mode = 0;       // SIMSTEP_HEAD_*
  int cost_transform = 0;  // SIMSTEP_COST_*

  TermConst term{};
  ImitConst* imit_dev = nullptr;
  void* policy = nullptr;  // PolicyStore (policy_api.inc)
  void* train = nullptr;   // TrainStore (train_api.inc)
  void* npg = nullptr;     // NpgStore (npg_api.inc)
  bool train_raw = false;  // tf32 handle in training: parameters keep all fp32 bits (they are the master copy)
  bool have_clip = false;
  int dof = 0;

  // optional per-category device timing (simstep_profile_*)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;   // begin/end pairs
  std::vector<int> prof_cat;
  int prof_open = -1;
  double prof_ms[SIMSTEP_PROF_CATEGORIES] = {0};
  long long prof_n[SIMSTEP_PROF_CATEGORIES] = {0};

  std::string err;
};

namespace {

// Brackets the launches issued while it is alive with two events on the launch stream.
struct ProfScope {
  simstep_handle* h;
  cudaStream_t st;
  bool on;
  ProfScope(simstep_handle* h_, int cat, cudaStream_t st_) : h(h_), st(st_), on(h_ && h_->prof_on) {
    if (!on) return;
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    h->prof_ev.push_back(a);
    h->prof_ev.push_back(b);
    h->prof_cat.push_back(cat);
    cudaEventRecord(a, st);
  }
  ~ProfScope() {
    if (on) cudaEventRecord(h->prof_ev.back(), st);
  }
};

// Makes `device` current for the lifetime of the object and restores the caller's device afterwards (the load_*
// entry points allocate on the handle's device but must not change the calling thread's current device).
struct DeviceScope {
  int prev = -1;
  explicit DeviceScope(int device) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != device) cudaSetDevice(device);
    else prev = -1;
  }
  ~DeviceScope() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int fail(simstep_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_error = msg;
  return code;
}

#define CU_TRY(h, expr)                                                                                   \
  do {                                                                                                    \
    cudaError_t e__ = (expr);                                                                             \
    if (e__ != cudaSuccess)                                                                               \
      return fail(h, SIMSTEP_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(e__) + " (" __FILE__ ":" + \
                                        std::to_string(__LINE__) + ")");                                 \
  } while (0)

// Launch with programmatic stream serialization (see ptx::grid_dep_wait): the kernel may be scheduled while the
// previous kernel of the stream drains; every kernel launched this way starts with grid_dep_wait().
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// K-major operand [rows][cols] with a (128-byte x box_rows) box and 128-byte swizzle.
int encode_operand(simstep_handle* h, CUtensorMap* map, int prec, void* base, long long cols, long long rows,
                   long long pitch_elems, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(h, SIMSTEP_ECUDA, "cuTensorMapEncodeTiled entry point not found");
  const int es = prec == SIMSTEP_PREC_TF32 ? 4 : 2;
  const CUtensorMapDataType dt = prec == SIMSTEP_PREC_TF32   ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : prec == SIMSTEP_PREC_FP16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                                             : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(pitch_elems) * es};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / es), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, dt, 2, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(h, SIMSTEP_ECUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(r)));
  return SIMSTEP_OK;
}

template <typename E, int MODE, int CG, int EG>
int launch_gemm_t(simstep_handle* h, const CUtensorMap& ax, const CUtensorMap& ah, const CUtensorMap& b,
                  const CUtensorMap& out, const GemmArgs& ga, int sm_count, cudaStream_t st) {
  static bool attr_set[kMaxDevices] = {};  // function attributes are per device
  auto kern = gemm_tcgen05_kernel<E, MODE, CG, EG>;
  using Plan = GemmPlan<CG, EG, !epi_is_rff(MODE)>;
  constexpr size_t smem = Plan::smem_bytes();
  int dev = h ? h->device : 0;  // h is null for simstep_debug_gemm: use the calling thread's current device
  if (!h) CU_TRY(h, cudaGetDevice(&dev));
  bool& attr_done = attr_set[dev % kMaxDevices];
  if (!attr_done) {
    CU_TRY(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    attr_done = true;
  }
  const int total = ga.m_tiles * ga.n_tiles * ga.groups;
  if (total <= 0) return SIMSTEP_OK;
  // persistent: one CTA (CG = 1) or one CTA pair (CG = 2) per tile slot, at most one CTA per SM
  const int n_inner = ga.n_inner > 1 ? ga.n_inner : 1;
  const int slots = std::min(total / n_inner, sm_count / CG);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(unsigned(slots * CG));
  cfg.blockDim = dim3(Plan::kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  CU_TRY(h, cudaLaunchKernelEx(&cfg, kern, ax, ah, b, out, ga));
  g_launches++;
  return SIMSTEP_OK;
}

// SIMSTEP_GEMM_WIDE_EPI=0: one epilogue group everywhere (the round-1 kernels), for A/B runs
bool wide_epilogue_enabled() {
  static const bool on = [] { const char* e = std::getenv("SIMSTEP_GEMM_WIDE_EPI"); return !(e && e[0] == '0'); }();
  return on;
}

template <int MODE>
int launch_gemm(simstep_handle* h, int prec, int cg, const CUtensorMap& ax, const CUtensorMap& ah, const CUtensorMap& b,
                const CUtensorMap& out, const GemmArgs& ga, int sm_count, cudaStream_t st) {
  // Two epilogue groups where the epilogue, not the MMAs, bounds a tile: the cost-feature modes (a cosine per
  // element, no store staging), and store modes whose whole K fits the shortened ring (the first layer).
  constexpr bool kStore = !epi_is_rff(MODE);
  const bool wide = wide_epilogue_enabled() && cg == 2 && MODE != kEpiFinal &&
                    (!kStore || ga.kb_x + ga.kb_h <= GemmPlan<2, 2, true>::kStages);
#define SIMSTEP_GEMM_CASE(ELEM)                                                                    \
  if constexpr (MODE != kEpiFinal) {                                                               \
    if (wide) return launch_gemm_t<ELEM, MODE, 2, 2>(h, ax, ah, b, out, ga, sm_count, st);          \
  }                                                                                                \
  return cg == 2 ? launch_gemm_t<ELEM, MODE, 2, 1>(h, ax, ah, b, out, ga, sm_count, st)             \
                 : launch_gemm_t<ELEM, MODE, 1, 1>(h, ax, ah, b, out, ga, sm_count, st)
  switch (prec) {
    case SIMSTEP_PREC_TF32: SIMSTEP_GEMM_CASE(ElemTF32);
    case SIMSTEP_PREC_FP16: SIMSTEP_GEMM_CASE(ElemF16);
    case SIMSTEP_PREC_BF16: SIMSTEP_GEMM_CASE(ElemBF16);
  }
#undef SIMSTEP_GEMM_CASE
  return fail(h, SIMSTEP_EINVAL, "unknown precision");
}

// CTAs per GEMM tile: pairs unless SIMSTEP_GEMM_CG=1 asks for single-CTA tiles (bring-up / A-B comparisons)
int gemm_cta_group() {
  const char* e = std::getenv("SIMSTEP_GEMM_CG");
  return (e && e[0] == '1') ? 1 : 2;
}

int grid_for(long long work_items, int threads, int sm_count) {
  long long g = (work_items + threads - 1) / threads;
  const long long cap = static_cast<long long>(sm_count) * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return static_cast<int>(g);
}

int pack_matrix(simstep_handle* h, int prec, const float* src_dev, int src_pitch, int rows, void* dst,
                long long dst_pitch, const PackSegs& segs, int mode, cudaStream_t st) {
  if (rows <= 0) return SIMSTEP_OK;
  switch (prec) {
    case SIMSTEP_PREC_TF32:
      pack_weight_kernel<ElemTF32><<<rows, 128, 0, st>>>(src_dev, src_pitch, rows, static_cast<float*>(dst),
                                                         dst_pitch, segs, mode);
      break;
    case SIMSTEP_PREC_FP16:
      pack_weight_kernel<ElemF16><<<rows, 128, 0, st>>>(src_dev, src_pitch, rows, static_cast<__half*>(dst),
                                                        dst_pitch, segs, mode);
      break;
    default:
      pack_weight_kernel<ElemBF16><<<rows, 128, 0, st>>>(src_dev, src_pitch, rows, static_cast<__nv_bfloat16*>(dst),
                                                         dst_pitch, segs, mode);
  }
  g_launches++;
  CU_TRY(h, cudaGetLastError());
  return SIMSTEP_OK;
}

constexpr size_t kGuardBytes = 64 * 1024;

cudaError_t ws_alloc_bytes(simstep_handle* h, void** p, size_t bytes) {
  if (!h->guards_on) return cudaMalloc(p, bytes);
  char* base = nullptr;
  cudaError_t e = cudaMalloc(&base, bytes + 2 * kGuardBytes);
  if (e != cudaSuccess) return e;
  cudaMemset(base, 0xA5, kGuardBytes);
  cudaMemset(base + kGuardBytes + bytes, 0xA5, kGuardBytes);
  *p = base + kGuardBytes;
  h->guard_allocs.emplace_back(*p, bytes);
  return cudaSuccess;
}
template <typename T>
cudaError_t ws_alloc(simstep_handle* h, T** p, size_t bytes) {
  return ws_alloc_bytes(h, reinterpret_cast<void**>(p), bytes);
}
void ws_free(simstep_handle* h, void* p) {
  if (!p) return;
  for (size_t i = 0; i < h->guard_allocs.size(); ++i)
    if (h->guard_allocs[i].first == p) {
      cudaFree(static_cast<char*>(p) - kGuardBytes);
      h->guard_allocs.erase(h->guard_allocs.begin() + i);
      return;
    }
  cudaFree(p);
}

void free_workspace(simstep_handle* h) {
  ws_free(h, h->xbuf); h->xbuf = nullptr;
  ws_free(h, h->hbuf); h->hbuf = nullptr;
  ws_free(h, h->dws); h->dws = nullptr;
  cudaFree(h->tickets); h->tickets = nullptr;
  cudaFree(h->chain_cnt); h->chain_cnt = nullptr;
  ws_free(h, h->rffin); h->rffin = nullptr;
  ws_free(h, h->rff_part); h->rff_part = nullptr;
  h->cap_rows = 0;
}

long long chunk_limit(const simstep_handle* h) {
  long long c = h->cfg.max_chunk_envs > 0 ? h->cfg.max_chunk_envs : 65536;
  return round_up(c, h->row_align);
}

// Workspace for `rows` env rows per pass (grown on demand, never shrunk).
int ensure_workspace(simstep_handle* h, long long rows) {
  rows = round_up(rows < 1 ? 1 : rows, h->row_align);
  if (rows > chunk_limit(h)) rows = chunk_limit(h);
  if (rows <= h->cap_rows && (!h->have_rff || h->rffin || (h->feat_net && h->rff_part))) return SIMSTEP_OK;
  if (rows < h->cap_rows) rows = h->cap_rows;
  CU_TRY(h, cudaDeviceSynchronize());
  free_workspace(h);
  const int prec = h->cfg.precision;
  if (h->have_ensemble || h->S > 0) {
    CU_TRY(h, ws_alloc(h, &h->xbuf, size_t(rows) * h->XP * h->esize));
    if (h->HT > 0) CU_TRY(h, ws_alloc(h, &h->hbuf, size_t(h->N) * rows * h->HT * h->esize));
    CU_TRY(h, ws_alloc(h, &h->dws, size_t(h->N) * rows * h->DP * sizeof(float)));
    CU_TRY(h, cudaMalloc(&h->tickets, size_t(rows / kBlockM + 2) * sizeof(unsigned int)));
    CU_TRY(h, cudaMemset(h->tickets, 0, size_t(rows / kBlockM + 2) * sizeof(unsigned int)));
    CU_TRY(h, cudaMalloc(&h->chain_cnt, size_t(h->sm_count) * 2 * sizeof(unsigned int)));
    CU_TRY(h, cudaMemset(h->chain_cnt, 0, size_t(h->sm_count) * 2 * sizeof(unsigned int)));
    CU_TRY(h, cudaMemset(h->xbuf, 0, size_t(rows) * h->XP * h->esize));
    if (h->HT > 0) CU_TRY(h, cudaMemset(h->hbuf, 0, size_t(h->N) * rows * h->HT * h->esize));
    int rc = encode_operand(h, &h->tmap_x, prec, h->xbuf, h->XP, rows, h->XP, kBlockM);
    if (rc) return rc;
    if (h->HT > 0) {
      rc = encode_operand(h, &h->tmap_h, prec, h->hbuf, h->HT, static_cast<long long>(h->N) * rows, h->HT, kBlockM);
      if (rc) return rc;
    } else {
      h->tmap_h = h->tmap_x;
    }
    // fp32 delta workspace, written by the final layer's TMA-store epilogue (32-float x 128-row boxes); the
    // map is DP columns wide, so the store clips the padded output columns instead of writing them
    rc = encode_operand(h, &h->tmap_dws, SIMSTEP_PREC_TF32, h->dws, h->DP, static_cast<long long>(h->N) * rows, h->DP,
                        kBlockM);
    if (rc) return rc;
  }
  if (h->have_rff && h->feat_net) {
    CU_TRY(h, ws_alloc(h, &h->rff_part, size_t(h->D_pad / kBlockN) * rows * sizeof(float)));  // A operand = hbuf
  } else if (h->have_rff) {
    const int rka = h->rff_split_cap ? 2 * h->RK : h->RK;  // [hi | lo]; the hi block is read twice by the GEMM
    CU_TRY(h, ws_alloc(h, &h->rffin, size_t(rows) * rka * h->esize));
    CU_TRY(h, cudaMemset(h->rffin, 0, size_t(rows) * rka * h->esize));
    CU_TRY(h, ws_alloc(h, &h->rff_part, size_t(h->D_pad / kBlockN) * rows * sizeof(float)));
    int rc = encode_operand(h, &h->tmap_rffin, prec, h->rffin, rka, rows, rka, kBlockM);
    if (rc) return rc;
  }
  h->cap_rows = rows;
  return SIMSTEP_OK;
}

template <typename E>
void launch_prep(simstep_handle* h, const float* s, const float* a, long long n, long long rows_pad,
                 const float* w_src, cudaStream_t st) {
  const int grid = int(std::min<long long>(rows_pad, static_cast<long long>(h->sm_count) * 16));
  // column pairs are read with one 8-byte load when no pair straddles the state / action boundary
  const bool vec = h->S % 2 == 0 && h->A % 2 == 0 && reinterpret_cast<uintptr_t>(s) % 8 == 0 &&
                   reinterpret_cast<uintptr_t>(a) % 8 == 0;
  auto kern = vec ? prep_input_kernel<E, true> : prep_input_kernel<E, false>;
  launch_pdl(kern, dim3(grid), dim3(kPrepThreads), 0, st, s, a, h->S, h->A, h->XP, n, rows_pad,
             h->cfg.transform ? h->tf_dev : nullptr, static_cast<typename E::storage*>(h->xbuf), w_src,
             w_src ? h->rff_wpad : nullptr, h->D, h->sat_dev);
  g_launches++;
}

// The env step's tail for a chunk (caller tensors, chunk-local row 0): given to run_ensemble_chunk it is fused into
// the final layer's launch (gemm_final.cuh) when final_fused_ok() says so; otherwise launch_post() runs it.
struct StepTail {
  const float* state = nullptr;
  float* next_state = nullptr;
  const int32_t* member = nullptr;
  int32_t* num_steps = nullptr;
  float* disc = nullptr;
  uint8_t* done = nullptr;
  bool rff = false;  // also write the cost features' operand rows of [s; s'] (input_type 'ss')
};

// SIMSTEP_FINAL_FUSED=1 selects the single-launch final layer + env-step tail (gemm_final.cuh).  It is correct
// (the parity suite passes with it) but NOT the default: measured on B200 it is slower than the final-layer GEMM
// followed by the post-step kernel (DESIGN.md section 5) - the final layer is HBM-bound, and the tails' L2 round
// trips queue behind the operand stream.
bool final_fused_enabled() {
  static const bool on = [] { const char* e = std::getenv("SIMSTEP_FINAL_FUSED"); return e && e[0] == '1'; }();
  return on;
}

bool final_fused_ok(const simstep_handle* h, const StepTail& t) {
  const Layer& fin = h->layers[h->L];
  return final_fused_enabled() && h->cg == 2 && h->S % 2 == 0 && h->S <= kBlockN && fin.o_pad == kBlockN &&
         reinterpret_cast<uintptr_t>(t.state) % 16 == 0 && reinterpret_cast<uintptr_t>(t.next_state) % 16 == 0 &&
         (t.next_state == nullptr || t.state != nullptr) && final_smem_bytes(h->S, h->N) <= 227 * 1024;
}

int launch_final(simstep_handle* h, long long n, long long rows_pad, const StepTail& t, cudaStream_t st) {
  const Layer& ly = h->layers[h->L];
  FinalLaunch fl;
  fl.ax = h->tmap_x;
  fl.ah = h->tmap_h;
  fl.b = ly.tmap_w;
  FinalArgs& fa = fl.args;
  fa = FinalArgs{};
  fa.m_tiles = int(rows_pad / (kBlockM * 2));
  fa.groups = h->N;
  fa.kb_x = ly.kb_x;
  fa.kb_h0 = ly.kb_h0;
  fa.kb_h = ly.kb_h;
  fa.a_rows_per_group = int(h->cap_rows);
  fa.b_rows_per_group = ly.o_pad;
  fa.bias = ly.bias;
  fa.scale = h->cfg.transform ? h->out_scale_dev : nullptr;
  fa.shift = h->cfg.transform ? h->out_shift_dev : nullptr;
  fa.dws_t = reinterpret_cast<float4*>(h->dws);
  fa.n_blocks = int(rows_pad / kBlockM);
  fa.counters = h->tickets;
  fa.state = t.state;
  fa.next_state = t.next_state;
  fa.member = t.member;
  fa.num_steps = t.num_steps;
  fa.disc = t.disc;
  fa.done = t.done;
  fa.n_rows = n;
  fa.S = h->S;
  fa.tc = h->term;
  if (t.rff) {
    fa.rff_out = h->rffin;
    fa.rff_pitch = h->rff_split_cap ? 2 * h->RK : h->RK;
    fa.rff_col2 = h->rff_col2;
    fa.rff_lo_off = h->rff_split ? h->RK : 0;
  }
  static const int dbg = [] { const char* e = std::getenv("SIMSTEP_FINAL_DEBUG"); return e ? std::atoi(e) : 0; }();
  fa.debug = dbg;
  CU_TRY(h, launch_final_fused(h->cfg.precision, fl, h->sm_count, h->device, st));
  g_launches++;
  return SIMSTEP_OK;
}

// The column-fused forward pass (gemm_chain.cuh): every layer of a (member, 256-row env tile) on one CTA pair, the
// activations handed from layer to layer through L2.  SIMSTEP_CHAIN=0 restores one launch per layer (A/B runs);
// SIMSTEP_CHAIN_SLOT=0 keeps the activation rows at their env rows instead of in the pair's L2-resident slot.
// SIMSTEP_CHAIN (A/B runs): 0 one launch per layer; 1 activation rows at their env rows instead of in the pair's
// L2-resident slot; 2 the default; 3 the last, partial round as a plain round instead of shared between pairs.
int chain_mode() {
  static const int mode = [] {
    const char* e = std::getenv("SIMSTEP_CHAIN");
    if (e && e[0] >= '0' && e[0] <= '3') return e[0] - '0';
    return 2;
  }();
  return mode;
}

// The chain kernel lives on L2 hits: every pair re-reads its unit's activation rows layer after layer while all members'
// weights stream past.  It is used while that working set - the packed weights plus one unit's [x | h] rows per CTA
// pair - fits 90 % of the L2 (108 of 126 MB at 4 x (512 x 4); measured 10 % faster than one launch per layer); an
// 8 x (1024 x 4) ensemble (136 MB of weights, 2.2 MB of activations per unit) thrashes it and was measured 14 % SLOWER,
// so such shapes keep one launch per layer.
// SIMSTEP_CHAIN_TAIL=1: the env step's tail (next state, discrepancy, termination, cost operand rows) runs INSIDE the
// chain kernel, on four extra warps per CTA, for the env tiles of its whole rounds but the last
// (SIMSTEP_CHAIN_TAIL_KEEP=<rounds left to the post-step kernel>, default 1).  Correct - next states, counters and masks
// bit-identical to the post-step kernel, the discrepancy within 2e-6 - and NOT the default: the chain kernel is bound by
// the L2->SM path its operands already saturate, so the tail's bytes cost there what they cost the post-step kernel
// outside (first round fused: launch +16 us, post-step kernel -18 us; all rounds: the last tiles' tails run after the
// MMAs have finished, +62 us against -36 us).
bool chain_tail_enabled() {
  static const bool on = [] { const char* e = std::getenv("SIMSTEP_CHAIN_TAIL"); return e && e[0] == '1'; }();
  return on;
}

bool chain_ok(const simstep_handle* h, long long rows_pad) {
  if (chain_mode() == 0 || h->cg != 2 || h->L < 1 || h->L + 1 > kChainMaxLayers || !h->have_ensemble) return false;
  static int l2_bytes[kMaxDevices] = {};
  int& l2 = l2_bytes[h->device % kMaxDevices];
  if (l2 == 0 && cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, h->device) != cudaSuccess) l2 = 1;
  double weights = 0;
  for (const Layer& ly : h->layers) weights += double(h->N) * ly.o_pad * ly.k_pad * h->esize;
  const long long units = rows_pad / (kBlockM * 2) * h->N;
  const double pairs = double(std::min<long long>(units, h->sm_count / 2));
  const double unit_bytes = double(kBlockM * 2) * (h->XP + h->HT) * h->esize;
  return weights + pairs * unit_bytes <= 0.9 * double(l2);
}

// The cost operand rows the step's tail also writes for input_type 'ss' (post kernels and the chain kernel's tail warps)
PostRff make_post_rff(const simstep_handle* h, bool fuse_rff) {
  PostRff rff{};
  if (fuse_rff) {
    rff.out = h->rffin;
    rff.prec = h->cfg.precision;
    rff.RK = h->RK;
    rff.split = h->rff_split;
    rff.col2 = h->rff_col2;
    rff.pitch = h->rff_split_cap ? 2 * h->RK : h->RK;
  }
  return rff;
}

int launch_chain(simstep_handle* h, long long rows_pad, cudaStream_t st, const StepTail* step_tail, long long n) {
  ChainLaunch cl;
  cl.maps.x = h->tmap_x;
  cl.maps.h = h->tmap_h;
  cl.maps.out_final = h->tmap_dws;
  ChainArgs& ca = cl.args;
  ca = ChainArgs{};
  ca.n_layers = h->L + 1;
  ca.m_tiles = int(rows_pad / (kBlockM * 2));
  ca.groups = h->N;
  ca.a_rows_per_group = int(h->cap_rows);
  ca.out_rows_per_group = int(h->cap_rows);
  ca.h_slot = chain_mode() == 1 ? 0 : 1;
  ca.scale = h->cfg.transform ? h->out_scale_dev : nullptr;
  ca.shift = h->cfg.transform ? h->out_shift_dev : nullptr;
  for (int l = 0; l <= h->L; ++l) {
    const Layer& ly = h->layers[l];
    cl.maps.w[l] = ly.tmap_w;
    ChainLayer& c = ca.layer[l];
    c.n_tiles = ly.o_pad / kBlockN;
    c.kb_x = ly.kb_x;
    c.kb_h0 = ly.kb_h0;
    c.kb_h = ly.kb_h;
    c.b_rows_per_group = ly.o_pad;
    c.out_col0 = ly.out_col0;
    c.bias = ly.bias;
    if (l < h->L) ca.hidden_tiles += c.n_tiles;
  }
  cl.maps.w_final64 = h->layers[h->L].tmap_w64;
  // L2 eviction priorities of the kernel's TMA traffic: weights and activations evict_last (every unit of a member
  // re-reads the same 5 MB of weights, a unit re-reads its own rows layer after layer), measured -2.5 % on the launch
  // (and +2.5 us on the post-step kernel, whose delta rows find less room in L2); marking x / the output evict_first
  // on top was measured neutral and is off.  SIMSTEP_CHAIN_HINTS=<mask> overrides for A/B runs.
  static const int hints = [] { const char* e = std::getenv("SIMSTEP_CHAIN_HINTS"); return e ? std::atoi(e) : 3; }();
  ca.l2_hints = hints;
  // the last, partial round: when its units are at most half the pairs, two pairs share each of them
  // whole rounds run with the members of an env tile in sequence on one pair: all pairs then stream the SAME member's
  // weights at any time (measured -1.5 % on the launch against members side by side; SIMSTEP_CHAIN_SEQ=0 for A/B)
  static const bool seq = [] { const char* e = std::getenv("SIMSTEP_CHAIN_SEQ"); return !(e && e[0] == '0'); }();
  int pairs = 1;
  chain_schedule(ca.m_tiles, ca.groups, h->sm_count / 2, seq,
                 chain_mode() != 3 && ca.hidden_tiles <= kChainMaxDepTiles && h->chain_cnt != nullptr, &pairs,
                 &ca.seq_rounds, &ca.tail_units);
  if (ca.tail_units > 0) {
    ca.tail_cnt = h->chain_cnt;
    int t = 0;
    for (int l = 0; l < h->L; ++l)
      for (int n = 0; n < ca.layer[l].n_tiles; ++n, ++t) {
        ca.dep_role[t] = static_cast<unsigned char>(n & 1);
        ca.dep_ord[t] = static_cast<unsigned char>(ca.tiles_per_role[n & 1]++);
      }
  }
  // The env step's tail inside this launch (gemm_chain.cuh, tail warps) for the env tiles of the whole rounds; the
  // post-step kernel then only gets the rows of the remaining units.
  static const int tail_keep = [] { const char* e = std::getenv("SIMSTEP_CHAIN_TAIL_KEEP"); return e ? std::atoi(e) : 1; }();
  const int tail_rounds = ca.seq_rounds - tail_keep;   // the last round's rows stay with the post-step kernel
  if (step_tail != nullptr && chain_tail_enabled() && tail_rounds > 0 && h->N == 4 && h->S % 2 == 0 &&
      h->S <= kPostMaxElems && reinterpret_cast<uintptr_t>(step_tail->state) % 8 == 0 &&
      reinterpret_cast<uintptr_t>(step_tail->next_state) % 8 == 0 && (step_tail->next_state == nullptr || step_tail->state != nullptr)) {
    ChainTail& t = ca.tail;
    t.enabled = 1;
    t.rounds = tail_rounds;
    t.delta = h->dws;
    t.delta_rows = h->cap_rows;
    t.DP = h->DP;
    t.state = step_tail->state;
    t.next_state = step_tail->next_state;
    t.member = step_tail->member;
    t.num_steps = step_tail->num_steps;
    t.disc = step_tail->disc;
    t.done = step_tail->done;
    t.n_rows = n;
    t.S = h->S;
    t.tc = h->term;
    t.rff = make_post_rff(h, step_tail->rff);
    h->tail_rows_done = std::min<long long>(n, static_cast<long long>(tail_rounds) * pairs * kBlockM * 2);
  }
  CU_TRY(h, launch_ensemble_chain(h->cfg.precision, h->cfg.activation != SIMSTEP_ACT_RELU, cl, h->sm_count, h->device, st));
  g_launches++;
  return SIMSTEP_OK;
}

// prep + all layer GEMMs for rows [0, n) of a chunk.  Without a tail (or when the tail cannot be fused) the
// un-normalised member deltas are left in h->dws[N][cap_rows][DP]; with a fusable tail the final layer's launch
// also runs the env step's tail and *tail_done is set.
// w_stage != nullptr: the prep kernel also copies the cost weights into h->rff_wpad (no separate memcpy node
// between the step's kernels).
int run_ensemble_chunk(simstep_handle* h, const float* s, const float* a, long long n, cudaStream_t st,
                       const float* w_stage = nullptr, int last_layer = -2, const StepTail* tail = nullptr,
                       bool* tail_done = nullptr) {
  if (last_layer == -2) last_layer = h->L;  // -1: input preparation only
  const long long rows_pad = round_up(n, h->row_align);
  if (tail_done) *tail_done = false;
  {
  ProfScope ps(h, SIMSTEP_PROF_PREP, st);
  switch (h->cfg.precision) {
    case SIMSTEP_PREC_TF32: launch_prep<ElemTF32>(h, s, a, n, rows_pad, w_stage, st); break;
    case SIMSTEP_PREC_FP16: launch_prep<ElemF16>(h, s, a, n, rows_pad, w_stage, st); break;
    default: launch_prep<ElemBF16>(h, s, a, n, rows_pad, w_stage, st);
  }
  }
  CU_TRY(h, cudaGetLastError());
  ProfScope ps(h, SIMSTEP_PROF_ENSEMBLE_GEMM, st);
  h->forward_was_chain = false;
  h->tail_rows_done = 0;
  if (last_layer == h->L && chain_ok(h, rows_pad) && !(tail != nullptr && final_fused_ok(h, *tail))) {
    h->forward_was_chain = true;
    return launch_chain(h, rows_pad, st, tail, n);
  }
  for (int l = 0; l <= last_layer; ++l) {
    const Layer& ly = h->layers[l];
    if (l == h->L && tail != nullptr && final_fused_ok(h, *tail)) {
      if (int rc = launch_final(h, n, rows_pad, *tail, st)) return rc;
      if (tail_done) *tail_done = true;
      break;
    }
    GemmArgs ga{};
    ga.m_tiles = int(rows_pad / (kBlockM * h->cg));
    ga.n_tiles = ly.o_pad / kBlockN;
    ga.groups = h->N;
    ga.kb_x = ly.kb_x;
    ga.kb_h0 = ly.kb_h0;
    ga.kb_h = ly.kb_h;
    ga.a_rows_per_group = int(h->cap_rows);
    ga.ax_rows_per_group = 0;
    ga.b_rows_per_group = ly.o_pad;
    ga.bias = ly.bias;
    ga.out_rows_per_group = int(h->cap_rows);
    // weight tiles with the evict_last L2 priority: every env tile of a member re-reads them while the activations
    // stream past (8 x (1024 x 4): -1 % on the five launches; neutral at 4 x (512 x 4); SIMSTEP_GEMM_B_HINT=0 for A/B)
    static const int b_hint = [] { const char* e = std::getenv("SIMSTEP_GEMM_B_HINT"); return e ? std::atoi(e) : 1; }();
    ga.b_evict_last = b_hint;
    int rc;
    if (l < h->L) {
      // bias + activation straight into this layer's K-slice of the concat buffer
      ga.out_col0 = ly.out_col0;
      rc = h->cfg.activation == SIMSTEP_ACT_RELU
               ? launch_gemm<kEpiHidden>(h, h->cfg.precision, h->cg, h->tmap_x, h->tmap_h, ly.tmap_w, h->tmap_h, ga,
                                         h->sm_count, st)
               : launch_gemm<kEpiHiddenTanh>(h, h->cfg.precision, h->cg, h->tmap_x, h->tmap_h, ly.tmap_w, h->tmap_h, ga,
                                             h->sm_count, st);
    } else {
      ga.out_col0 = 0;
      ga.scale = h->cfg.transform ? h->out_scale_dev : nullptr;
      ga.shift = h->cfg.transform ? h->out_shift_dev : nullptr;
      // the final layer is HBM-bound (every member re-reads its whole concat row for 226 outputs): run the members
      // of an env tile side by side (x comes from HBM once) and start with the rows whose last hidden slice the
      // previous launch wrote last (still in L2).  SIMSTEP_FINAL_ORDER=0 restores the plain order for A/B runs.
      static const bool order = [] { const char* e = std::getenv("SIMSTEP_FINAL_ORDER"); return !(e && e[0] == '0'); }();
      ga.group_fastest = order ? 1 : 0;
      ga.reverse = order ? 1 : 0;
      rc = launch_gemm<kEpiFinal>(h, h->cfg.precision, h->cg, h->tmap_x, h->tmap_h, ly.tmap_w, h->tmap_dws, ga,
                                  h->sm_count, st);
    }
    if (rc) return rc;
  }
  return SIMSTEP_OK;
}

// fuse_rff: also write the RFF operand rows of [s; s'] (input_type 'ss'), replacing rff_pack_kernel
int launch_post(simstep_handle* h, const float* state, const int32_t* member, int32_t* num_steps, long long n,
                float* next_state, float* disc, uint8_t* done, cudaStream_t st, bool fuse_rff = false) {
  if (h->S > kPostMaxElems) return fail(h, SIMSTEP_EINVAL, "state_dim > 256 is not supported by the post kernel");
  // rows whose tail already ran inside the chain kernel (launch_chain) are skipped: everything below is offset by row0
  const long long row0 = h->tail_rows_done;
  h->tail_rows_done = 0;
  if (row0 >= n) return SIMSTEP_OK;
  if (row0 > 0) {
    n -= row0;
    if (state) state += row0 * h->S;
    if (member) member += row0;
    if (num_steps) num_steps += row0;
    if (next_state) next_state += row0 * h->S;
    if (disc) disc += row0;
    if (done) done += row0;
  }
  const float* dws_base = h->dws + row0 * h->DP;
  ProfScope ps(h, SIMSTEP_PROF_POST, st);
  // one warp per row and one row per warp: the block scheduler balances the tail, no grid-stride quantisation
  const int blocks = int(std::min<long long>((n + kPostWarps - 1) / kPostWarps, 1LL << 30));
  const size_t smem = size_t(kPostWarps) * ((h->S + 3) & ~3) * sizeof(float);
  // float2 lanes need 8-byte aligned rows: even S and 8-byte aligned base pointers
  const bool vec2 = (h->S % 2 == 0) && (reinterpret_cast<uintptr_t>(state) % 8 == 0) &&
                    (reinterpret_cast<uintptr_t>(next_state) % 8 == 0);
  if (fuse_rff && !vec2) return fail(h, SIMSTEP_EINVAL, "internal: fused RFF operand needs the float2 path");
  PostRff rff = make_post_rff(h, fuse_rff);
  if (rff.out != nullptr) rff.out = static_cast<char*>(rff.out) + size_t(row0) * rff.pitch * h->esize;
  // TMA-staged persistent kernel (post_tma.cuh) whenever rows pair up into 16-byte granular spans
  const PostTmaPlan plan = post_tma_plan(h->S, h->DP, h->N);
  static const bool tma_off = [] { const char* e = std::getenv("SIMSTEP_POST_TMA"); return e && e[0] == '0'; }();
  const bool tma = !tma_off && plan.ok && vec2 && state != nullptr && next_state != nullptr &&
                   reinterpret_cast<uintptr_t>(state) % 16 == 0;
  // the chain kernel writes the deltas in row order: the last rows are the ones still in L2, so the rows are walked
  // backwards (SIMSTEP_POST_REVERSE=0: A/B); the per-layer final GEMM itself runs backwards, its LAST rows are row 0's
  static const int post_reverse_on = [] { const char* e = std::getenv("SIMSTEP_POST_REVERSE"); return (e && e[0] == '0') ? 0 : 1; }();
  const int post_reverse = (post_reverse_on && h->forward_was_chain) ? 1 : 0;
#define POST_TMA_LAUNCH(NM, ET)                                                                                \
  do {                                                                                                         \
    auto kern = h->S == 226 ? post_step_tma_kernel<NM, ET, 226> : post_step_tma_kernel<NM, ET, 0>;             \
    static size_t attr_smem[kMaxDevices][2] = {};  /* function attributes are per device */                   \
    size_t& attr_ref = attr_smem[h->device % kMaxDevices][h->S == 226 ? 1 : 0];                                                                               \
    if (attr_ref < plan.smem) {                                                                                \
      CU_TRY(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(plan.smem)));      \
      attr_ref = plan.smem;                                                                                    \
    }                                                                                                          \
    const long long pairs = (n + 1) / 2;                                                                       \
    const int grid = int(std::min<long long>((pairs + plan.rings - 1) / plan.rings, h->sm_count));             \
    launch_pdl(kern, dim3(grid), dim3(plan.rings * 64), plan.smem, st, dws_base, h->cap_rows, h->DP, state, member, \
               num_steps, h->S, n, next_state, disc, done, h->term, rff, plan.stages, post_reverse);           \
  } while (0)
#define POST_CASE(NM)                                                                                          \
  case NM:                                                                                                     \
    if (tma) {                                                                                                 \
      if (rff.out == nullptr || h->cfg.precision == SIMSTEP_PREC_FP16) POST_TMA_LAUNCH(NM, ElemF16);           \
      else if (h->cfg.precision == SIMSTEP_PREC_TF32) POST_TMA_LAUNCH(NM, ElemTF32);                           \
      else POST_TMA_LAUNCH(NM, ElemBF16);                                                                      \
    } else if (vec2)                                                                                           \
      launch_pdl(post_step_kernel<NM, 2>, dim3(blocks), dim3(kPostWarps * 32), smem, st, dws_base, h->cap_rows, h->DP, \
                 state, member, num_steps, h->S, n, next_state, disc, done, h->term, rff);                      \
    else                                                                                                       \
      launch_pdl(post_step_kernel<NM, 1>, dim3(blocks), dim3(kPostWarps * 32), smem, st, dws_base, h->cap_rows, h->DP, \
                 state, member, num_steps, h->S, n, next_state, disc, done, h->term, rff);                      \
    break;
  switch (h->N) {
    POST_CASE(1) POST_CASE(2) POST_CASE(3) POST_CASE(4) POST_CASE(5) POST_CASE(6) POST_CASE(7) POST_CASE(8)
    default: return fail(h, SIMSTEP_EINVAL, "n_models must be in [1, 8]");
  }
#undef POST_CASE
#undef POST_TMA_LAUNCH
  g_launches++;
  CU_TRY(h, cudaGetLastError());
  return SIMSTEP_OK;
}

int launch_rff_pack(simstep_handle* h, const RffSrc& src, long long n, cudaStream_t st) {
  ProfScope ps(h, SIMSTEP_PROF_RFF_PACK, st);
  const long long rows_pad = round_up(n, h->row_align);
  const int grid = int(std::min<long long>(rows_pad, static_cast<long long>(h->sm_count) * 16));
  const int pitch = h->rff_split_cap ? 2 * h->RK : h->RK;
  switch (h->cfg.precision) {
    case SIMSTEP_PREC_TF32:
      launch_pdl(rff_pack_kernel<ElemTF32>, dim3(grid), dim3(kPrepThreads), 0, st, src, h->RK, h->rff_split, pitch, n,
                 rows_pad, static_cast<float*>(h->rffin));
      break;
    case SIMSTEP_PREC_FP16:
      launch_pdl(rff_pack_kernel<ElemF16>, dim3(grid), dim3(kPrepThreads), 0, st, src, h->RK, h->rff_split, pitch, n,
                 rows_pad, static_cast<__half*>(h->rffin));
      break;
    default:
      launch_pdl(rff_pack_kernel<ElemBF16>, dim3(grid), dim3(kPrepThreads), 0, st, src, h->RK, h->rff_split, pitch, n,
                 rows_pad, static_cast<__nv_bfloat16*>(h->rffin));
  }
  g_launches++;
  CU_TRY(h, cudaGetLastError());
  return SIMSTEP_OK;
}

// What happens to a row's feature dot product (see CombineArgs).
CombineArgs make_combine(const simstep_handle* h, const float* disc, float lambda_b, float threshold, float c_min,
                         float c_max, int clamp_cost, float* dot, float* cost, float* ipm, float* bonus) {
  CombineArgs c{};
  c.enabled = 1;
  c.disc = disc;
  c.lambda_b = lambda_b;
  c.threshold = threshold;
  c.c_min = c_min;
  c.c_max = c_max;
  c.clamp_cost = clamp_cost;
  c.transform = h->cost_transform;
  c.dot_scale = (h->feat_net && h->feat_mode == SIMSTEP_HEAD_LINEAR) ? 1.f : float(std::sqrt(2.0 / h->D));
  c.dot_out = dot;
  c.cost = cost;
  c.ipm = ipm;
  c.bonus = bonus;
  return c;
}

// SIMSTEP_RFF_FUSED_COMBINE=0: partial dots per n-tile + cost_combine_kernel (the round-1 sequence), for A/B runs
bool rff_fused_combine() {
  static const bool on = [] { const char* e = std::getenv("SIMSTEP_RFF_FUSED_COMBINE"); return !(e && e[0] == '0'); }();
  return on;
}

// RFF GEMM over the packed rows of the chunk.  w_pad == nullptr: features only.  comb != nullptr: the epilogue
// finishes cost / ipm / bonus itself (a CTA pair then runs all n-tiles of its rows back to back and carries the dot
// product in registers); otherwise the per-n-tile partial dots go to h->rff_part for cost_combine_kernel.
int launch_rff_gemm(simstep_handle* h, long long n, const float* w_pad, float* phi, cudaStream_t st,
                    const CombineArgs* comb = nullptr) {
  ProfScope ps(h, SIMSTEP_PROF_RFF_GEMM, st);
  GemmArgs ga{};
  ga.m_tiles = int(round_up(n, h->row_align) / (kBlockM * h->cg));
  ga.n_tiles = h->D_pad / kBlockN;
  ga.groups = 1;
  // K loop: [hi | lo] through the first map, then the hi block again (x_hi * W_lo) through the second; without the
  // split only the hi block (the first RK columns of the row operand and of the packed weight)
  ga.kb_x = (h->rff_split ? 2 * h->RK : h->RK) / h->bk;
  ga.kb_h0 = 0;
  ga.kb_h = h->rff_split ? h->RK / h->bk : 0;
  ga.a_rows_per_group = 0;
  ga.b_rows_per_group = h->D_pad;
  ga.bias = h->rff_b;
  ga.scale = w_pad;
  ga.out = phi;
  ga.out_pitch = h->D;
  ga.rows_valid = int(n);
  ga.cols_valid = h->D;
  ga.rff_part = w_pad ? h->rff_part : nullptr;
  ga.rff_part_stride = h->cap_rows;
  ga.rff_phi_scale = float(std::sqrt(2.0 / h->D));
  if (comb != nullptr && w_pad != nullptr) {
    ga.comb = *comb;
    ga.n_inner = ga.n_tiles;
    ga.rff_part = nullptr;
  }
  if (h->feat_net) {
    // the head reads the last hidden layer's slice of the activation buffer
    const Layer& fin = h->layers[h->L];
    ga.kb_x = fin.kb_x;   // no hidden layer: the head reads the input rows themselves
    ga.kb_h0 = fin.kb_h0;
    ga.kb_h = fin.kb_h;
    ga.rff_tanh = h->feat_mode == SIMSTEP_HEAD_TANH_COS;
    ga.rff_linear = h->feat_mode == SIMSTEP_HEAD_LINEAR;
    if (ga.rff_linear) ga.rff_phi_scale = 1.f;
    return launch_gemm<kEpiFeat>(h, h->cfg.precision, h->cg, h->tmap_x, h->tmap_h, h->tmap_rffw, h->tmap_h, ga,
                                h->sm_count, st);
  }
  return launch_gemm<kEpiRff>(h, h->cfg.precision, h->cg, h->tmap_rffin, h->tmap_rffin, h->tmap_rffw, h->tmap_rffin, ga,
                              h->sm_count, st);
}

// RFF GEMM + bonus combine for the packed rows of a chunk (one launch, or two with SIMSTEP_RFF_FUSED_COMBINE=0)
int launch_rff_cost(simstep_handle* h, long long n, const CombineArgs& comb, cudaStream_t st) {
  if (rff_fused_combine()) return launch_rff_gemm(h, n, h->rff_wpad, nullptr, st, &comb);
  if (int rc = launch_rff_gemm(h, n, h->rff_wpad, nullptr, st)) return rc;
  ProfScope ps(h, SIMSTEP_PROF_COMBINE, st);
  launch_pdl(cost_combine_kernel, dim3(grid_for(n, 256, h->sm_count)), dim3(256), 0, st, h->rff_part, h->cap_rows,
             h->D_pad / kBlockN, n, comb);
  g_launches++;
  CU_TRY(h, cudaGetLastError());
  return SIMSTEP_OK;
}

int stage_w(simstep_handle* h, const float* w_dev, cudaStream_t st) {
  CU_TRY(h, cudaMemcpyAsync(h->rff_wpad, w_dev, size_t(h->D) * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return SIMSTEP_OK;
}

// Operand-row sources for the cost features of (s, a, s').  Operand columns follow the reference's concatenation
// order (linear_cost.py:115-126) except for input_type 'ss', where s' starts at column rff_col2 (see load_rff).
int rff_sources(simstep_handle* h, const float* s, const float* a, const float* s2, RffSrc* out) {
  RffSrc r{};
  const int S = h->S, A = h->A, in = h->rff_in;
  auto seg = [&](const float* p, int width, int pitch, int dst0) {
    r.ptr[r.n] = p; r.width[r.n] = width; r.pitch[r.n] = pitch; r.dst0[r.n] = dst0; r.n++;
  };
  if (in == 2 * S && s2) { seg(s, S, S, 0); seg(s2, S, S, h->rff_col2); }
  else if (in == S) { seg(s, S, S, 0); }
  else if (in == S + A) { seg(s, S, S, 0); seg(a, A, A, S); }
  else if (in == 2 * S + A && s2) { seg(s, S, S, 0); seg(a, A, A, S); seg(s2, S, S, S + A); }
  else return fail(h, SIMSTEP_EINVAL, "rff in_dim does not match an input_type of s/ss/sa/sas");
  *out = r;
  return SIMSTEP_OK;
}

// Operand-row source for explicit feature-input rows x [n][rff_in] (get_rep / get_costs on caller-built inputs).
RffSrc rff_row_source(const simstep_handle* h, const float* x) {
  RffSrc r{};
  const int in = h->rff_in;
  if (h->rff_col2 > 0) {  // 'ss' layout: the two halves of a row go to columns 0 and rff_col2
    const int half = in / 2;
    r.n = 2;
    r.ptr[0] = x; r.width[0] = half; r.pitch[0] = in; r.dst0[0] = 0;
    r.ptr[1] = x + half; r.width[1] = half; r.pitch[1] = in; r.dst0[1] = h->rff_col2;
  } else {
    r.n = 1;
    r.ptr[0] = x; r.width[0] = in; r.pitch[0] = in; r.dst0[0] = 0;
  }
  return r;
}

// Packs layer l of every member (weights_host[m * stride + l], nn.Linear layout) into the operand format.
int upload_layer(simstep_handle* h, int l, const float* const* weights_host, const float* const* biases_host,
                 int stride) {
  cudaStream_t st = nullptr;
  Layer& ly = h->layers[l];
  const size_t wbytes = size_t(h->N) * ly.o_pad * ly.k_pad * h->esize;
  if (!ly.w) CU_TRY(h, cudaMalloc(&ly.w, wbytes));
  if (!ly.bias) CU_TRY(h, cudaMalloc(&ly.bias, size_t(h->N) * ly.o_pad * sizeof(float)));
  CU_TRY(h, cudaMemsetAsync(ly.w, 0, wbytes, st));
  CU_TRY(h, cudaMemsetAsync(ly.bias, 0, size_t(h->N) * ly.o_pad * sizeof(float), st));
  float* tmp = nullptr;
  CU_TRY(h, cudaMalloc(&tmp, size_t(ly.out) * ly.in_ref * sizeof(float)));
  for (int m = 0; m < h->N; ++m) {
    const float* wsrc = weights_host[m * stride + l];
    const float* bsrc = biases_host[m * stride + l];
    if (!wsrc || !bsrc) { cudaFree(tmp); return fail(h, SIMSTEP_EINVAL, "null weight or bias pointer"); }
    CU_TRY(h, cudaMemcpyAsync(tmp, wsrc, size_t(ly.out) * ly.in_ref * sizeof(float), cudaMemcpyHostToDevice, st));
    void* dst = static_cast<char*>(ly.w) + size_t(m) * ly.o_pad * ly.k_pad * h->esize;
    int rc = pack_matrix(h, h->cfg.precision, tmp, ly.in_ref, ly.out, dst, ly.k_pad, ly.segs, h->train_raw ? 3 : 0, st);
    if (rc) { cudaFree(tmp); return rc; }
    CU_TRY(h, cudaMemcpyAsync(ly.bias + size_t(m) * ly.o_pad, bsrc, size_t(ly.out) * sizeof(float),
                              cudaMemcpyHostToDevice, st));
    CU_TRY(h, cudaStreamSynchronize(st));  // tmp and the pageable host source are reused
  }
  cudaFree(tmp);
  if (int rc = encode_operand(h, &ly.tmap_w64, h->cfg.precision, ly.w, ly.k_pad, static_cast<long long>(h->N) * ly.o_pad,
                              ly.k_pad, kBlockN / 4))
    return rc;
  return encode_operand(h, &ly.tmap_w, h->cfg.precision, ly.w, ly.k_pad, static_cast<long long>(h->N) * ly.o_pad,
                        ly.k_pad, kBlockN / h->cg);
}

void free_clip(simstep_handle* h);
void free_policy(simstep_handle* h);
void free_train(simstep_handle* h);
void free_npg(simstep_handle* h);

// A handle's buffers, tensor maps and kernel attributes belong to the device it was created on; work can only be
// enqueued from a thread whose current device is that one (one process per GPU does this by construction).
int check_device(simstep_handle* h) {
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess || dev != h->device)
    return fail(h, SIMSTEP_EINVAL, "the handle was created on device " + std::to_string(h->device) +
                                       " but the calling thread's current device is " + std::to_string(dev));
  return SIMSTEP_OK;
}

int check_step_ready(simstep_handle* h, long long n_envs) {
  if (!h) return SIMSTEP_EINVAL;
  if (int rc = check_device(h)) return rc;
  if (h->feat_net) return fail(h, SIMSTEP_EINVAL, "this handle holds a cost feature net, not a dynamics ensemble");
  if (!h->have_ensemble) return fail(h, SIMSTEP_EINVAL, "simstep_load_ensemble has not been called");
  if (n_envs < 0) return fail(h, SIMSTEP_EINVAL, "n_envs < 0");
  return SIMSTEP_OK;
}

}  // namespace

// =============================================================================

extern "C" {

int simstep_abi_version(void) { return SIMSTEP_ABI_VERSION; }

const char* simstep_last_error(const simstep_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int64_t simstep_launch_count(void) { return g_launches.load(); }

int simstep_create(const simstep_config* cfg, simstep_handle** out) {
  if (!cfg || !out) return fail(nullptr, SIMSTEP_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->abi_version != SIMSTEP_ABI_VERSION) return fail(nullptr, SIMSTEP_EINVAL, "abi_version mismatch");
  if (cfg->state_dim < 1 || cfg->action_dim < 0 || cfg->n_models < 1 || cfg->n_models > 8 || cfg->n_hidden < 0 ||
      cfg->n_hidden > SIMSTEP_MAX_HIDDEN)
    return fail(nullptr, SIMSTEP_EINVAL, "bad ensemble shape");
  if (cfg->precision < 0 || cfg->precision > 2) return fail(nullptr, SIMSTEP_EINVAL, "bad precision");
  for (int i = 0; i < cfg->n_hidden; ++i)
    if (cfg->hidden[i] < 1) return fail(nullptr, SIMSTEP_EINVAL, "bad hidden size");
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return fail(nullptr, SIMSTEP_ENODEV, std::string("cudaGetDevice: ") + cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return fail(nullptr, SIMSTEP_ENODEV, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, SIMSTEP_ENODEV,
                "libsimstep is built for sm_100a only; device is sm_" + std::to_string(prop.major * 10 + prop.minor));

  simstep_handle* h = new simstep_handle();
  h->cfg = *cfg;
  h->device = dev;
  h->sm_count = prop.multiProcessorCount;
  h->esize = cfg->precision == SIMSTEP_PREC_TF32 ? 4 : 2;
  h->bk = 128 / h->esize;
  h->cg = gemm_cta_group();
  { const char* e = std::getenv("SIMSTEP_DEBUG_GUARDS"); h->guards_on = e && e[0] == '1'; }
  h->row_align = kBlockM * h->cg;
  h->S = cfg->state_dim;
  h->A = cfg->action_dim;
  h->N = cfg->n_models;
  h->L = cfg->n_hidden;
  h->XP = int(round_up(h->S + h->A, 64));
  h->SP = int(round_up(h->S, kBlockN));
  h->DP = int(round_up(h->S, 4));
  std::vector<int> hp(h->L), hcol(h->L);
  int ht = 0;
  for (int i = 0; i < h->L; ++i) {
    hp[i] = int(round_up(cfg->hidden[i], kBlockN));
    hcol[i] = ht;
    ht += hp[i];
  }
  h->HT = ht;
  h->layers.resize(h->L + 1);
  const int X = h->S + h->A;
  for (int l = 0; l <= h->L; ++l) {
    Layer& ly = h->layers[l];
    ly.out = l < h->L ? cfg->hidden[l] : h->S;
    ly.o_pad = l < h->L ? hp[l] : h->SP;
    ly.out_col0 = l < h->L ? hcol[l] : 0;
    PackSegs& sg = ly.segs;
    sg.n = 0;
    if (cfg->dense_connect || l == 0) {
      // K order of BasicMLP's concat: [x, h_1, ..., h_l]  (dynamics.py:414-419, 427-430)
      ly.kb_x = h->XP / h->bk;
      sg.src0[0] = 0; sg.width[0] = X; sg.dst0[0] = 0; sg.n = 1;
      int src = X;
      for (int j = 0; j < l && cfg->dense_connect; ++j) {
        sg.src0[sg.n] = src; sg.width[sg.n] = cfg->hidden[j]; sg.dst0[sg.n] = h->XP + hcol[j];
        src += cfg->hidden[j];
        sg.n++;
      }
      ly.in_ref = src;
      ly.kb_h0 = 0;
      ly.kb_h = (cfg->dense_connect && l > 0) ? (hcol[l - 1] + hp[l - 1]) / h->bk : 0;
      ly.k_pad = h->XP + ly.kb_h * h->bk;
    } else {
      ly.kb_x = 0;
      ly.kb_h0 = hcol[l - 1] / h->bk;
      ly.kb_h = hp[l - 1] / h->bk;
      ly.k_pad = hp[l - 1];
      ly.in_ref = cfg->hidden[l - 1];
      sg.src0[0] = 0; sg.width[0] = cfg->hidden[l - 1]; sg.dst0[0] = 0; sg.n = 1;
    }
  }
  if (cudaMalloc(&h->sat_dev, sizeof(unsigned long long)) != cudaSuccess ||
      cudaMemset(h->sat_dev, 0, sizeof(unsigned long long)) != cudaSuccess) {
    delete h;
    return fail(nullptr, SIMSTEP_ENOMEM, "cudaMalloc failed");
  }
  // default termination model: none (horizon only) until simstep_set_termination
  h->term.horizon = 300;
  h->term.vel_inv_divisor = 1.f;
  h->term.vel_threshold = 100.f;
  h->term.pos_dim = 3;
  *out = h;
  return SIMSTEP_OK;
}

int simstep_destroy(simstep_handle* h) {
  if (!h) return SIMSTEP_OK;
  cudaDeviceSynchronize();
  free_workspace(h);
  for (auto& ly : h->layers) {
    cudaFree(ly.w);
    cudaFree(ly.bias);
  }
  cudaFree(h->sat_dev);
  cudaFree(h->tf_dev);
  cudaFree(h->out_scale_dev);
  cudaFree(h->out_shift_dev);
  cudaFree(h->rff_w);
  cudaFree(h->rff_b);
  cudaFree(h->rff_wpad);
  cudaFree(h->colsum_partial);
  free_clip(h);
  free_npg(h);
  free_policy(h);
  free_train(h);
  delete h;
  return SIMSTEP_OK;
}

int simstep_query(const simstep_handle* h, int32_t* n_layers, int32_t* layer_in, int32_t* layer_out,
                  int64_t* chunk_envs, int64_t* workspace_bytes) {
  if (!h) return SIMSTEP_EINVAL;
  if (n_layers) *n_layers = h->L + 1;
  for (int l = 0; l <= h->L; ++l) {
    if (layer_in) layer_in[l] = h->layers[l].in_ref;
    if (layer_out) layer_out[l] = h->layers[l].out;
  }
  if (chunk_envs) *chunk_envs = chunk_limit(h);
  if (workspace_bytes) {
    const long long r = h->cap_rows;
    *workspace_bytes = r * h->XP * h->esize + static_cast<long long>(h->N) * r * h->HT * h->esize +
                       static_cast<long long>(h->N) * r * h->DP * 4 + (h->have_rff ? r * (h->rff_split_cap ? 2 * h->RK : h->RK) * h->esize : 0);
  }
  return SIMSTEP_OK;
}

int simstep_load_ensemble(simstep_handle* h, const float* const* weights_host, const float* const* biases_host,
                          const float* const* transforms_host) {
  if (!h || !weights_host || !biases_host) return fail(h, SIMSTEP_EINVAL, "null argument");
  if (h->cfg.transform && !transforms_host) return fail(h, SIMSTEP_EINVAL, "transform set but no transforms given");
  DeviceScope dev_scope(h->device);  // parameters live on the handle's device; the caller's current device is restored
  const int nl = h->L + 1;
  for (int l = 0; l < nl; ++l) {
    int rc = upload_layer(h, l, weights_host, biases_host, nl);
    if (rc) return rc;
  }
  // transforms
  const int S = h->S, A = h->A;
  if (!h->tf_dev) CU_TRY(h, cudaMalloc(&h->tf_dev, size_t(2 * S + 2 * A + 4) * sizeof(float)));
  if (!h->out_scale_dev) CU_TRY(h, cudaMalloc(&h->out_scale_dev, size_t(h->SP) * sizeof(float)));
  if (!h->out_shift_dev) CU_TRY(h, cudaMalloc(&h->out_shift_dev, size_t(h->SP) * sizeof(float)));
  if (h->cfg.transform) {
    for (int i = 0; i < 6; ++i)
      if (!transforms_host[i]) return fail(h, SIMSTEP_EINVAL, "null transform vector");
    std::vector<float> tf(2 * S + 2 * A), osc(h->SP, 1.f), osh(h->SP, 0.f);
    std::memcpy(tf.data(), transforms_host[0], S * sizeof(float));
    std::memcpy(tf.data() + S, transforms_host[1], S * sizeof(float));
    std::memcpy(tf.data() + 2 * S, transforms_host[2], A * sizeof(float));
    std::memcpy(tf.data() + 2 * S + A, transforms_host[3], A * sizeof(float));
    std::memcpy(osh.data(), transforms_host[4], S * sizeof(float));
    std::memcpy(osc.data(), transforms_host[5], S * sizeof(float));
    CU_TRY(h, cudaMemcpy(h->tf_dev, tf.data(), tf.size() * sizeof(float), cudaMemcpyHostToDevice));
    CU_TRY(h, cudaMemcpy(h->out_scale_dev, osc.data(), osc.size() * sizeof(float), cudaMemcpyHostToDevice));
    CU_TRY(h, cudaMemcpy(h->out_shift_dev, osh.data(), osh.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  CU_TRY(h, cudaDeviceSynchronize());
  h->have_ensemble = true;
  return SIMSTEP_OK;
}

int simstep_set_termination(simstep_handle* h, const simstep_termination* t) {
  if (!h || !t) return fail(h, SIMSTEP_EINVAL, "null argument");
  if (t->n_bodies < 0 || t->n_bodies > SIMSTEP_MAX_BODIES) return fail(h, SIMSTEP_EINVAL, "bad n_bodies");
  TermConst& c = h->term;
  c.horizon = t->horizon;
  c.enable_velocity_check = t->enable_velocity_check;
  c.vel_offset = t->vel_offset;
  c.vel_threshold = t->vel_threshold;
  c.vel_inv_divisor = t->vel_divisor != 0.f ? 1.f / t->vel_divisor : 1.f;
  c.record_all_world = t->record_all_world;
  c.record_world_root_pos = t->record_world_root_pos;
  c.n_bodies = t->n_bodies;
  c.pos_dim = t->pos_dim > 0 ? t->pos_dim : 3;
  for (int i = 0; i < t->n_bodies; ++i) {
    if (t->body_offset[i] < 0 || t->body_offset[i] + c.pos_dim + 1 >= h->S)
      return fail(h, SIMSTEP_EINVAL, "body offset outside the state vector");
    c.body_offset[i] = t->body_offset[i];
    c.body_shape[i] = t->body_shape[i];
    c.body_radius[i] = 0.5f * t->body_param0[i];
    c.body_half_height[i] = 0.5f * t->body_param1[i];
  }
  return SIMSTEP_OK;
}

int simstep_load_rff(simstep_handle* h, int32_t feature_dim, int32_t in_dim, const float* weight_host,
                     const float* bias_host, int32_t split) {
  if (!h || !weight_host || !bias_host || feature_dim < 1 || in_dim < 1) return fail(h, SIMSTEP_EINVAL, "bad argument");
  DeviceScope dev_scope(h->device);  // parameters live on the handle's device; the caller's current device is restored
  CU_TRY(h, cudaDeviceSynchronize());
  cudaFree(h->rff_w); cudaFree(h->rff_b); cudaFree(h->rff_wpad); cudaFree(h->colsum_partial);
  ws_free(h, h->rffin); ws_free(h, h->rff_part);
  h->rff_w = nullptr; h->rff_b = nullptr; h->rff_wpad = nullptr; h->colsum_partial = nullptr;
  h->rffin = nullptr; h->rff_part = nullptr;
  h->have_rff = false;
  h->D = feature_dim;
  h->D_pad = int(round_up(feature_dim, kBlockN));
  h->rff_in = in_dim;
  // input_type 'ss' on an ensemble handle (in_dim == 2 S): s' starts at column S rounded up to 8 instead of S, so the
  // step's fused tail writes both halves of an operand row with aligned 16-byte stores; weight columns follow
  h->rff_col2 = (h->S > 0 && in_dim == 2 * h->S && !h->feat_net) ? int(round_up(h->S, 8)) : 0;
  h->RK = int(round_up(h->rff_col2 > 0 ? h->rff_col2 + h->S : in_dim, 64));
  h->rff_split_cap = split ? 1 : 0;
  h->rff_split = h->rff_split_cap;
  h->RKT = h->rff_split_cap ? 3 * h->RK : h->RK;  // K of the packed weight; the row operand stores 2*RK
  const size_t wbytes = size_t(h->D_pad) * h->RKT * h->esize;
  CU_TRY(h, cudaMalloc(&h->rff_w, wbytes));
  CU_TRY(h, cudaMemset(h->rff_w, 0, wbytes));
  CU_TRY(h, cudaMalloc(&h->rff_b, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMemset(h->rff_b, 0, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMalloc(&h->rff_wpad, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMemset(h->rff_wpad, 0, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMalloc(&h->colsum_partial, size_t(1024) * h->D_pad * sizeof(double)));
  float* tmp = nullptr;
  CU_TRY(h, cudaMalloc(&tmp, size_t(feature_dim) * in_dim * sizeof(float)));
  CU_TRY(h, cudaMemcpy(tmp, weight_host, size_t(feature_dim) * in_dim * sizeof(float), cudaMemcpyHostToDevice));
  CU_TRY(h, cudaMemcpy(h->rff_b, bias_host, size_t(feature_dim) * sizeof(float), cudaMemcpyHostToDevice));
  PackSegs sg{};
  sg.n = 1; sg.src0[0] = 0; sg.width[0] = in_dim;
  if (h->rff_col2 > 0) {
    sg.n = 2; sg.width[0] = h->S;
    sg.src0[1] = h->S; sg.width[1] = h->S;
  }
  // operand triple on the A side is [hi | lo | hi]; B side is [hi | hi | lo]
  const int modes[3] = {1, 1, 2};
  for (int part = 0; part < (h->rff_split_cap ? 3 : 1); ++part) {
    sg.dst0[0] = part * h->RK;
    sg.dst0[1] = part * h->RK + h->rff_col2;
    int rc = pack_matrix(h, h->cfg.precision, tmp, in_dim, feature_dim, h->rff_w, h->RKT, sg,
                         h->rff_split_cap ? modes[part] : 0, nullptr);
    if (rc) { cudaFree(tmp); return rc; }
  }
  CU_TRY(h, cudaDeviceSynchronize());
  cudaFree(tmp);
  int rc = encode_operand(h, &h->tmap_rffw, h->cfg.precision, h->rff_w, h->RKT, h->D_pad, h->RKT, kBlockN / h->cg);
  if (rc) return rc;
  h->have_rff = true;
  return SIMSTEP_OK;
}

int simstep_load_feature_net(simstep_handle* h, const float* const* weights_host, const float* const* biases_host,
                             int32_t feature_dim, const float* head_weight_host, const float* head_bias_host,
                             int32_t head_mode) {
  if (!h || !weights_host || !biases_host || !head_weight_host || !head_bias_host || feature_dim < 1)
    return fail(h, SIMSTEP_EINVAL, "bad argument");
  if (head_mode != SIMSTEP_HEAD_TANH_COS && head_mode != SIMSTEP_HEAD_LINEAR)
    return fail(h, SIMSTEP_EINVAL, "head_mode must be SIMSTEP_HEAD_TANH_COS or SIMSTEP_HEAD_LINEAR");
  if (h->N != 1 || h->A != 0 || h->cfg.transform || h->cfg.dense_connect)
    return fail(h, SIMSTEP_EINVAL,
                "a feature net needs a handle with n_models = 1, action_dim = 0, transform = 0 and dense_connect = 0");
  DeviceScope dev_scope(h->device);  // parameters live on the handle's device; the caller's current device is restored
  CU_TRY(h, cudaDeviceSynchronize());
  for (int l = 0; l < h->L; ++l) {
    int rc = upload_layer(h, l, weights_host, biases_host, h->L);
    if (rc) return rc;
  }
  if (!h->tf_dev) CU_TRY(h, cudaMalloc(&h->tf_dev, size_t(2 * h->S + 4) * sizeof(float)));
  // head = cos-feature layer over the last hidden activations (reuses the random-feature GEMM epilogue)
  cudaFree(h->rff_w); cudaFree(h->rff_b); cudaFree(h->rff_wpad); cudaFree(h->colsum_partial);
  ws_free(h, h->rffin); ws_free(h, h->rff_part);
  h->rff_w = nullptr; h->rff_b = nullptr; h->rff_wpad = nullptr; h->colsum_partial = nullptr;
  h->rffin = nullptr; h->rff_part = nullptr;
  h->have_rff = false;
  const Layer& fin = h->layers[h->L];
  const int in_dim = h->L > 0 ? h->cfg.hidden[h->L - 1] : h->S;
  h->D = feature_dim;
  h->D_pad = int(round_up(feature_dim, kBlockN));
  h->rff_in = in_dim;
  h->RK = (fin.kb_x + fin.kb_h) * h->bk;  // the padded width of the last hidden layer's slice (or of the input)
  h->rff_split = 0;
  h->rff_split_cap = 0;
  h->rff_col2 = 0;
  h->RKT = h->RK;
  const size_t wbytes = size_t(h->D_pad) * h->RKT * h->esize;
  CU_TRY(h, cudaMalloc(&h->rff_w, wbytes));
  CU_TRY(h, cudaMemset(h->rff_w, 0, wbytes));
  CU_TRY(h, cudaMalloc(&h->rff_b, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMemset(h->rff_b, 0, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMalloc(&h->rff_wpad, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMemset(h->rff_wpad, 0, size_t(h->D_pad) * sizeof(float)));
  CU_TRY(h, cudaMalloc(&h->colsum_partial, size_t(1024) * h->D_pad * sizeof(double)));
  float* tmp = nullptr;
  CU_TRY(h, cudaMalloc(&tmp, size_t(feature_dim) * in_dim * sizeof(float)));
  CU_TRY(h, cudaMemcpy(tmp, head_weight_host, size_t(feature_dim) * in_dim * sizeof(float), cudaMemcpyHostToDevice));
  CU_TRY(h, cudaMemcpy(h->rff_b, head_bias_host, size_t(feature_dim) * sizeof(float), cudaMemcpyHostToDevice));
  PackSegs sg{};
  sg.n = 1; sg.src0[0] = 0; sg.width[0] = in_dim; sg.dst0[0] = 0;
  int rc = pack_matrix(h, h->cfg.precision, tmp, in_dim, feature_dim, h->rff_w, h->RKT, sg, 0, nullptr);
  CU_TRY(h, cudaDeviceSynchronize());
  cudaFree(tmp);
  if (rc) return rc;
  rc = encode_operand(h, &h->tmap_rffw, h->cfg.precision, h->rff_w, h->RKT, h->D_pad, h->RKT, kBlockN / h->cg);
  if (rc) return rc;
  free_workspace(h);
  h->feat_mode = head_mode;
  h->feat_net = true;
  h->have_rff = true;
  h->have_ensemble = true;
  return SIMSTEP_OK;
}

int simstep_set_cost_transform(simstep_handle* h, int32_t transform) {
  if (!h) return SIMSTEP_EINVAL;
  if (transform < SIMSTEP_COST_IDENTITY || transform > SIMSTEP_COST_GAIL_LL) return fail(h, SIMSTEP_EINVAL, "bad cost transform");
  h->cost_transform = transform;
  return SIMSTEP_OK;
}

int simstep_saturation_count(simstep_handle* h, int64_t* count_out, int32_t reset) {
  if (!h || !count_out) return fail(h, SIMSTEP_EINVAL, "null argument");
  unsigned long long v = 0;
  CU_TRY(h, cudaMemcpy(&v, h->sat_dev, sizeof(v), cudaMemcpyDeviceToHost));  // synchronises with the device
  if (reset) CU_TRY(h, cudaMemset(h->sat_dev, 0, sizeof(v)));
  *count_out = static_cast<int64_t>(v);
  return SIMSTEP_OK;
}

int simstep_debug_check_guards(simstep_handle* h, int64_t* buffers_out, int64_t* bad_bytes_out) {
  if (!h || !buffers_out || !bad_bytes_out) return fail(h, SIMSTEP_EINVAL, "null argument");
  *buffers_out = static_cast<int64_t>(h->guard_allocs.size());
  *bad_bytes_out = 0;
  if (!h->guards_on) return SIMSTEP_OK;
  CU_TRY(h, cudaDeviceSynchronize());
  std::vector<unsigned char> host(kGuardBytes);
  for (const auto& g : h->guard_allocs) {
    const char* user = static_cast<const char*>(g.first);
    const char* zones[2] = {user - kGuardBytes, user + g.second};
    for (const char* z : zones) {
      CU_TRY(h, cudaMemcpy(host.data(), z, kGuardBytes, cudaMemcpyDeviceToHost));
      for (unsigned char b : host) *bad_bytes_out += b != 0xA5;
    }
  }
  return SIMSTEP_OK;
}

int simstep_debug_chain_schedule(int32_t m_tiles, int32_t groups, int32_t sm_count, int32_t max_items,
                                 int32_t* pairs_out, int32_t* seq_rounds_out, int32_t* tail_units_out,
                                 int32_t* items_out) {
  if (m_tiles < 1 || groups < 1 || sm_count < 2 || max_items < 1 || !pairs_out || !seq_rounds_out || !tail_units_out ||
      !items_out)
    return SIMSTEP_EINVAL;
  ChainArgs a{};
  a.m_tiles = m_tiles;
  a.groups = groups;
  int pairs = 1;
  chain_schedule(m_tiles, groups, sm_count / 2, true, true, &pairs, &a.seq_rounds, &a.tail_units);
  *pairs_out = pairs;
  *seq_rounds_out = a.seq_rounds;
  *tail_units_out = a.tail_units;
  for (int p = 0; p < pairs; ++p) {
    int32_t* row = items_out + static_cast<size_t>(p) * max_items * 2;
    ChainItem it;
    int i = 0;
    for (; chain_item(a, p, pairs, i, it); ++i) {
      if (i >= max_items - 1) return SIMSTEP_EINVAL;
      row[2 * i] = it.unit;
      row[2 * i + 1] = it.role;
    }
    row[2 * i] = -1;      // terminator
    row[2 * i + 1] = -1;
  }
  return SIMSTEP_OK;
}

int simstep_forward_launches(const simstep_handle* h, int64_t n_envs, int32_t* launches_out) {
  if (!h || !launches_out || n_envs < 1) return SIMSTEP_EINVAL;
  const long long rows = std::min<long long>(round_up(n_envs, h->row_align), chunk_limit(h));
  *launches_out = chain_ok(h, rows) && !final_fused_enabled() ? 1 : h->L + 1;
  return SIMSTEP_OK;
}

int simstep_set_rff_split(simstep_handle* h, int32_t split) {
  if (!h) return SIMSTEP_EINVAL;
  if (!h->have_rff || h->feat_net) return fail(h, SIMSTEP_EINVAL, "simstep_load_rff has not been called");
  if (split && !h->rff_split_cap)
    return fail(h, SIMSTEP_EINVAL, "the random-feature layer was loaded without hi/lo operand pairs (split = 0)");
  h->rff_split = split ? 1 : 0;
  return SIMSTEP_OK;
}

int simstep_forward(simstep_handle* h, const float* state_dev, const float* action_dev, int64_t n_envs,
                    float* delta_dev, void* stream) {
  int rc = check_step_ready(h, n_envs);
  if (rc) return rc;
  if (n_envs == 0) return SIMSTEP_OK;
  if (!state_dev || !action_dev || !delta_dev) return fail(h, SIMSTEP_EINVAL, "null device pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = ensure_workspace(h, n_envs))) return rc;
  for (long long r0 = 0; r0 < n_envs; r0 += h->cap_rows) {
    const long long n = std::min<long long>(h->cap_rows, n_envs - r0);
    if ((rc = run_ensemble_chunk(h, state_dev + r0 * h->S, action_dev + r0 * h->A, n, st))) return rc;
    const long long total = static_cast<long long>(h->N) * n * h->S;
    extract_delta_kernel<<<grid_for(total, 256, h->sm_count), 256, 0, st>>>(h->dws, h->cap_rows, h->DP, h->N, h->S, n,
                                                                            delta_dev, n_envs, r0);
    g_launches++;
    CU_TRY(h, cudaGetLastError());
  }
  return SIMSTEP_OK;
}

int simstep_discrepancy(simstep_handle* h, const float* state_dev, const float* action_dev, int64_t n_envs,
                        float* disc_dev, void* stream) {
  int rc = check_step_ready(h, n_envs);
  if (rc) return rc;
  if (n_envs == 0) return SIMSTEP_OK;
  if (!state_dev || !action_dev || !disc_dev) return fail(h, SIMSTEP_EINVAL, "null device pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = ensure_workspace(h, n_envs))) return rc;
  for (long long r0 = 0; r0 < n_envs; r0 += h->cap_rows) {
    const long long n = std::min<long long>(h->cap_rows, n_envs - r0);
    StepTail tail;
    tail.disc = disc_dev + r0;
    bool tail_done = false;
    if ((rc = run_ensemble_chunk(h, state_dev + r0 * h->S, action_dev + r0 * h->A, n, st, nullptr, -2, &tail, &tail_done)))
      return rc;
    if (!tail_done && (rc = launch_post(h, nullptr, nullptr, nullptr, n, nullptr, disc_dev + r0, nullptr, st))) return rc;
  }
  return SIMSTEP_OK;
}

int simstep_step(simstep_handle* h, const float* state_dev, const float* action_dev, const int32_t* member_dev,
                 int32_t* num_steps_dev, int64_t n_envs, float* next_state_dev, float* disc_dev, uint8_t* done_dev,
                 void* stream) {
  int rc = check_step_ready(h, n_envs);
  if (rc) return rc;
  if (n_envs == 0) return SIMSTEP_OK;
  if (!state_dev || !action_dev || !next_state_dev) return fail(h, SIMSTEP_EINVAL, "null device pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = ensure_workspace(h, n_envs))) return rc;
  for (long long r0 = 0; r0 < n_envs; r0 += h->cap_rows) {
    const long long n = std::min<long long>(h->cap_rows, n_envs - r0);
    StepTail tail;
    tail.state = state_dev + r0 * h->S;
    tail.next_state = next_state_dev + r0 * h->S;
    tail.member = member_dev ? member_dev + r0 : nullptr;
    tail.num_steps = num_steps_dev ? num_steps_dev + r0 : nullptr;
    tail.disc = disc_dev ? disc_dev + r0 : nullptr;
    tail.done = done_dev ? done_dev + r0 : nullptr;
    bool tail_done = false;
    if ((rc = run_ensemble_chunk(h, tail.state, action_dev + r0 * h->A, n, st, nullptr, -2, &tail, &tail_done))) return rc;
    if (!tail_done && (rc = launch_post(h, tail.state, tail.member, tail.num_steps, n, tail.next_state, tail.disc,
                                        tail.done, st)))
      return rc;
  }
  return SIMSTEP_OK;
}

int simstep_step_cost(simstep_handle* h, const float* state_dev, const float* action_dev, const int32_t* member_dev,
                      int32_t* num_steps_dev, int64_t n_envs, float* next_state_dev, float* disc_dev,
                      uint8_t* done_dev, const float* w_dev, float lambda_b, float threshold, float c_min, float c_max,
                      int32_t clamp_cost, float* cost_dev, float* ipm_dev, float* bonus_dev, void* stream) {
  int rc = check_step_ready(h, n_envs);
  if (rc) return rc;
  if (!h->have_rff) return fail(h, SIMSTEP_EINVAL, "simstep_load_rff has not been called");
  if (n_envs == 0) return SIMSTEP_OK;
  if (!state_dev || !action_dev || !next_state_dev || !disc_dev || !w_dev)
    return fail(h, SIMSTEP_EINVAL, "null device pointer (state, action, next_state, disc and w are required)");
  if (next_state_dev == state_dev) return fail(h, SIMSTEP_EINVAL, "next_state must not alias state in step_cost");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((rc = ensure_workspace(h, n_envs))) return rc;
  for (long long r0 = 0; r0 < n_envs; r0 += h->cap_rows) {
    const long long n = std::min<long long>(h->cap_rows, n_envs - r0);
    const float* s = state_dev + r0 * h->S;
    const float* a = action_dev + r0 * h->A;
    float* s2 = next_state_dev + r0 * h->S;
    // input_type 'ss' with float2-able rows: the step's tail writes the cost features' operand rows itself
    const bool fuse = h->rff_col2 > 0 && h->S % 2 == 0 && reinterpret_cast<uintptr_t>(s) % 8 == 0 &&
                      reinterpret_cast<uintptr_t>(s2) % 8 == 0;
    StepTail tail;
    tail.state = s;
    tail.next_state = s2;
    tail.member = member_dev ? member_dev + r0 : nullptr;
    tail.num_steps = num_steps_dev ? num_steps_dev + r0 : nullptr;
    tail.disc = disc_dev + r0;
    tail.done = done_dev ? done_dev + r0 : nullptr;
    tail.rff = fuse;
    bool tail_done = false;
    if ((rc = run_ensemble_chunk(h, s, a, n, st, r0 == 0 ? w_dev : nullptr, -2, &tail, &tail_done))) return rc;
    if (!tail_done &&
        (rc = launch_post(h, s, tail.member, tail.num_steps, n, s2, tail.disc, tail.done, st, fuse)))
      return rc;
    if (!fuse) {
      RffSrc src;
      if ((rc = rff_sources(h, s, a, s2, &src))) return rc;
      if ((rc = launch_rff_pack(h, src, n, st))) return rc;
    }
    const CombineArgs comb = make_combine(h, disc_dev + r0, lambda_b, threshold, c_min, c_max, clamp_cost, nullptr,
                                          cost_dev ? cost_dev + r0 : nullptr, ipm_dev ? ipm_dev + r0 : nullptr,
                                          bonus_dev ? bonus_dev + r0 : nullptr);
    if ((rc = launch_rff_cost(h, n, comb, st))) return rc;
  }
  return SIMSTEP_OK;
}

int simstep_rff_features(simstep_handle* h, const float* x_dev, int64_t n_rows, float* phi_dev, double* phi_sum_dev,
                         void* stream) {
  if (!h) return SIMSTEP_EINVAL;
  if (!h->have_rff) return fail(h, SIMSTEP_EINVAL, "simstep_load_rff has not been called");
  if (int rc0 = check_device(h)) return rc0;
  if (n_rows < 0 || (n_rows > 0 && (!x_dev || !phi_dev))) return fail(h, SIMSTEP_EINVAL, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if (n_rows > 0) {
    if ((rc = ensure_workspace(h, n_rows))) return rc;
    for (long long r0 = 0; r0 < n_rows; r0 += h->cap_rows) {
      const long long n = std::min<long long>(h->cap_rows, n_rows - r0);
      if (h->feat_net) {
        if ((rc = run_ensemble_chunk(h, x_dev + r0 * h->S, nullptr, n, st, nullptr, h->L - 1))) return rc;
      } else {
        if ((rc = launch_rff_pack(h, rff_row_source(h, x_dev + r0 * h->rff_in), n, st))) return rc;
      }
      if ((rc = launch_rff_gemm(h, n, nullptr, phi_dev + r0 * h->D, st))) return rc;
    }
  }
  if (phi_sum_dev) {
    const int nb = int(std::min<long long>(1024, std::max<long long>(1, (n_rows + 63) / 64)));
    const int rpb = int((n_rows + nb - 1) / nb);
    colsum_partial_kernel<<<nb, 256, 0, st>>>(phi_dev, n_rows, h->D, rpb > 0 ? rpb : 1, h->colsum_partial);
    colsum_final_kernel<<<(h->D + 255) / 256, 256, 0, st>>>(h->colsum_partial, nb, h->D, phi_sum_dev, 0);
    g_launches += 2;
    CU_TRY(h, cudaGetLastError());
  }
  return SIMSTEP_OK;
}

int simstep_rff_dot(simstep_handle* h, const float* x_dev, int64_t n_rows, const float* w_dev, float* dot_dev,
                    void* stream) {
  return simstep_bonus_cost(h, x_dev, nullptr, n_rows, w_dev, 0.f, 1.f, 0.f, 0.f, 0, dot_dev, nullptr, nullptr,
                            stream);
}

int simstep_bonus_cost(simstep_handle* h, const float* x_dev, const float* disc_dev, int64_t n_rows,
                       const float* w_dev, float lambda_b, float threshold, float c_min, float c_max,
                       int32_t clamp_cost, float* cost_dev, float* ipm_dev, float* bonus_dev, void* stream) {
  if (!h) return SIMSTEP_EINVAL;
  if (!h->have_rff) return fail(h, SIMSTEP_EINVAL, "simstep_load_rff has not been called");
  if (int rc0 = check_device(h)) return rc0;
  if (n_rows < 0) return fail(h, SIMSTEP_EINVAL, "n_rows < 0");
  if (n_rows == 0) return SIMSTEP_OK;
  if (!x_dev || !w_dev) return fail(h, SIMSTEP_EINVAL, "null device pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc;
  if ((rc = ensure_workspace(h, n_rows))) return rc;
  if ((rc = stage_w(h, w_dev, st))) return rc;
  for (long long r0 = 0; r0 < n_rows; r0 += h->cap_rows) {
    const long long n = std::min<long long>(h->cap_rows, n_rows - r0);
    if (h->feat_net) {
      if ((rc = run_ensemble_chunk(h, x_dev + r0 * h->S, nullptr, n, st, nullptr, h->L - 1))) return rc;
    } else {
      if ((rc = launch_rff_pack(h, rff_row_source(h, x_dev + r0 * h->rff_in), n, st))) return rc;
    }
    // disc_dev == nullptr (simstep_rff_dot): cost_dev receives the raw phi . w
    const CombineArgs comb =
        disc_dev == nullptr
            ? make_combine(h, nullptr, 0.f, 1.f, 0.f, 0.f, 0, cost_dev ? cost_dev + r0 : nullptr, nullptr, nullptr, nullptr)
            : make_combine(h, disc_dev + r0, lambda_b, threshold, c_min, c_max, clamp_cost, nullptr,
                           cost_dev ? cost_dev + r0 : nullptr, ipm_dev ? ipm_dev + r0 : nullptr,
                           bonus_dev ? bonus_dev + r0 : nullptr);
    if ((rc = launch_rff_cost(h, n, comb, st))) return rc;
  }
  return SIMSTEP_OK;
}

int simstep_reduce_max_sum(simstep_handle* h, const float* x_dev, int64_t n, double* out_dev, void* stream) {
  if (!h || !out_dev || n < 0 || (n > 0 && !x_dev)) return fail(h, SIMSTEP_EINVAL, "bad argument");
  reduce_max_sum_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(x_dev, n, out_dev);
  g_launches++;
  CU_TRY(h, cudaGetLastError());
  return SIMSTEP_OK;
}

int simstep_profile_enable(simstep_handle* h, int32_t enable) {
  if (!h) return SIMSTEP_EINVAL;
  h->prof_on = enable != 0;
  return SIMSTEP_OK;
}

int simstep_profile_read(simstep_handle* h, double* ms_out, int64_t* count_out, int32_t reset) {
  if (!h) return SIMSTEP_EINVAL;
  CU_TRY(h, cudaDeviceSynchronize());
  for (size_t i = 0; i < h->prof_cat.size(); ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]) == cudaSuccess) {
      h->prof_ms[h->prof_cat[i]] += ms;
      h->prof_n[h->prof_cat[i]] += 1;
    }
    cudaEventDestroy(h->prof_ev[2 * i]);
    cudaEventDestroy(h->prof_ev[2 * i + 1]);
  }
  h->prof_ev.clear();
  h->prof_cat.clear();
  for (int c = 0; c < SIMSTEP_PROF_CATEGORIES; ++c) {
    if (ms_out) ms_out[c] = h->prof_ms[c];
    if (count_out) count_out[c] = h->prof_n[c];
    if (reset) { h->prof_ms[c] = 0; h->prof_n[c] = 0; }
  }
  return SIMSTEP_OK;
}

int simstep_debug_gemm(int32_t precision, int32_t groups, int64_t m, int32_t n, int32_t k, const float* a_dev,
                       const float* b_dev, const float* bias_dev, float* d_dev, void* stream) {
  if (precision < 0 || precision > 2 || groups < 1 || m < 1 || n < 1 || k < 1 || !a_dev || !b_dev || !d_dev)
    return fail(nullptr, SIMSTEP_EINVAL, "bad argument");
  simstep_handle* h = nullptr;  // errors go to the create-error slot
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int cg = gemm_cta_group();
  const int es = precision == SIMSTEP_PREC_TF32 ? 4 : 2;
  const int bk = 128 / es;
  const long long m_pad = round_up(m, kBlockM * cg), n_pad = round_up(n, kBlockN), k_pad = round_up(k, 64);
  cudaDeviceProp prop;
  int dev = 0;
  CU_TRY(h, cudaGetDevice(&dev));
  CU_TRY(h, cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(nullptr, SIMSTEP_ENODEV, "libsimstep is built for sm_100a only");
  void *ap = nullptr, *bp = nullptr;
  float *biasp = nullptr, *dp = nullptr;  // dp: padded fp32 output [groups][m_pad][n_pad] of the TMA-store epilogue
  CU_TRY(h, cudaMalloc(&ap, size_t(groups) * m_pad * k_pad * es));
  CU_TRY(h, cudaMalloc(&bp, size_t(groups) * n_pad * k_pad * es));
  CU_TRY(h, cudaMalloc(&biasp, size_t(groups) * n_pad * sizeof(float)));
  CU_TRY(h, cudaMalloc(&dp, size_t(groups) * m_pad * n_pad * sizeof(float)));
  CU_TRY(h, cudaMemsetAsync(ap, 0, size_t(groups) * m_pad * k_pad * es, st));
  CU_TRY(h, cudaMemsetAsync(bp, 0, size_t(groups) * n_pad * k_pad * es, st));
  CU_TRY(h, cudaMemsetAsync(biasp, 0, size_t(groups) * n_pad * sizeof(float), st));
  PackSegs sg{};
  sg.n = 1; sg.src0[0] = 0; sg.width[0] = k; sg.dst0[0] = 0;
  int rc = SIMSTEP_OK;
  for (int g = 0; g < groups && !rc; ++g) {
    rc = pack_matrix(h, precision, a_dev + size_t(g) * m * k, k, int(m), static_cast<char*>(ap) + size_t(g) * m_pad * k_pad * es,
                     k_pad, sg, 0, st);
    if (!rc)
      rc = pack_matrix(h, precision, b_dev + size_t(g) * n * k, k, n, static_cast<char*>(bp) + size_t(g) * n_pad * k_pad * es,
                       k_pad, sg, 0, st);
    if (!rc && bias_dev)
      if (cudaMemcpyAsync(biasp + size_t(g) * n_pad, bias_dev + size_t(g) * n, size_t(n) * sizeof(float),
                          cudaMemcpyDeviceToDevice, st) != cudaSuccess)
        rc = fail(nullptr, SIMSTEP_ECUDA, "bias copy failed");
  }
  if (!rc) {
    cudaError_t pe = cudaStreamSynchronize(st);
    if (pe != cudaSuccess) rc = fail(nullptr, SIMSTEP_ECUDA, std::string("debug gemm pack stage: ") + cudaGetErrorString(pe));
  }
  CUtensorMap ta, tb, td;
  if (!rc) rc = encode_operand(h, &ta, precision, ap, k_pad, groups * m_pad, k_pad, kBlockM);
  if (!rc) rc = encode_operand(h, &tb, precision, bp, k_pad, groups * n_pad, k_pad, kBlockN / cg);
  if (!rc) rc = encode_operand(h, &td, SIMSTEP_PREC_TF32, dp, n_pad, groups * m_pad, n_pad, kBlockM);
  if (!rc) {
    GemmArgs ga{};
    ga.m_tiles = int(m_pad / (kBlockM * cg));
    ga.n_tiles = int(n_pad / kBlockN);
    ga.groups = groups;
    ga.kb_x = 0;
    ga.kb_h0 = 0;
    ga.kb_h = int(k_pad / bk);
    ga.a_rows_per_group = int(m_pad);
    ga.b_rows_per_group = int(n_pad);
    ga.bias = biasp;
    ga.out_rows_per_group = int(m_pad);
    ga.out_col0 = 0;
    rc = launch_gemm<kEpiFinal>(h, precision, cg, ta, ta, tb, td, ga, prop.multiProcessorCount, st);
  }
  if (!rc) {
    const long long total = static_cast<long long>(groups) * m * n;
    extract_delta_kernel<<<grid_for(total, 256, prop.multiProcessorCount), 256, 0, st>>>(dp, m_pad, int(n_pad), groups, n,
                                                                                         m, d_dev, m, 0);
    g_launches++;
  }
  cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(ap);
  cudaFree(bp);
  cudaFree(biasp);
  cudaFree(dp);
  if (!rc && e != cudaSuccess) return fail(nullptr, SIMSTEP_ECUDA, std::string("debug gemm: ") + cudaGetErrorString(e));
  return rc;
}

}  // extern "C"

#include "imitation_api.inc"
#include "policy_api.inc"
#include "train_api.inc"
#include "npg_api.inc"
