// C ABI of libvitocm.so (see include/vitocm.h).  Host-side engine: weight store + repack,
// TMA tensor-map construction, kernel launches.  No torch types; plain pointers and sizes.
#include "../../include/vitocm.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "attention_bwd_sm100.cuh"
#include "attention_sm100.cuh"
#include "gemm_sm100.cuh"
#include "attention_quad_sm100.cuh"
#include "mlp_fused_sm100.cuh"
#include "block_tail_sm100.cuh"
#include "post_kernels.cuh"
#include "train_kernels.cuh"
#include "vit_kernels.cuh"
#include "wgrad_sm100.cuh"

using namespace vitocm;

namespace {

thread_local char g_err[512] = "";
std::atomic<long long> g_launches{0};

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CUDA_TRY(expr)                                                                                      \
  do {                                                                                                      \
    cudaError_t err__ = (expr);                                                                             \
    if (err__ != cudaSuccess) return fail(VITOCM_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(err__), __FILE__, __LINE__); \
  } while (0)
#define TRY(expr)                \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != 0) return rc__;  \
  } while (0)
#define LAUNCH_CHECK()                                                                                            \
  do {                                                                                                            \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                                           \
    cudaError_t err__ = cudaGetLastError();                                                                       \
    if (err__ != cudaSuccess) return fail(VITOCM_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(err__), __FILE__, __LINE__); \
  } while (0)

// ---- optional per-kernel-class device timing (CUDA events on the launching stream) ----
enum ProfClass { PC_PATCH = 0, PC_LN, PC_GEMM_QKV, PC_ATTN, PC_GEMM_PROJ, PC_GEMM_FC1, PC_GEMM_FC2, PC_GEMM_KLAST, PC_CLSROW,
                 PC_POST, PC_OTHER, PC_WGRAD, PC_DGRAD, PC_ATTN_BWD, PC_TRAIN_ELEM, PC_OPTIM, PC_MLP, PC_TAIL, PC_COUNT };
const char* const kProfNames[PC_COUNT] = {"patch_embed", "layernorm", "gemm_qkv", "attention", "gemm_proj", "gemm_fc1_gelu",
                                          "gemm_fc2", "gemm_k_last", "cls_attn_row", "post", "other", "gemm_wgrad", "gemm_dgrad",
                                          "attention_bwd", "train_elementwise", "optimizer", "mlp_fused", "block_tail"};
struct ProfRec { int cls; cudaEvent_t a, b; };
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
struct ProfScope {
  cudaStream_t st; bool on; ProfRec r;
  ProfScope(int cls, cudaStream_t s) : st(s), on(g_prof_on) {
    if (on) { r.cls = cls; cudaEventCreate(&r.a); cudaEventCreate(&r.b); cudaEventRecord(r.a, st); }
  }
  ~ProfScope() { if (on) { cudaEventRecord(r.b, st); g_prof.push_back(r); } }
};

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda link dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// Tensor map over a dense row-major matrix (rank 2: [rows][ld]; rank 3: [outer][rows][ld] with `outer_stride`
// elements between slabs).  Operand loads: bf16, box [box_rows][64], SWIZZLE_128B.  Epilogue stores: box
// [32][32], SWIZZLE_64B (bf16) or SWIZZLE_128B (fp32).
int make_tmap(CUtensorMap* tm, const void* ptr, bool f32, long long cols, long long rows, long long ld, int box_cols,
              int box_rows, CUtensorMapSwizzle swz, long long outer = 0, long long outer_stride = 0) {
  EncodeTiledFn fn = get_encode_fn();
  if (fn == nullptr) return fail(VITOCM_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const int es = f32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld * es) % 16 != 0 || (outer_stride * es) % 16 != 0)
    return fail(VITOCM_ERR_INVALID, "TMA operand must be 16-byte aligned with a 16-byte multiple row pitch");
  const cuuint32_t rank = outer > 0 ? 3 : 2;
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(outer)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(ld) * es, static_cast<cuuint64_t>(outer_stride) * es};
  cuuint32_t box[3] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows), 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = fn(tm, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(ptr), dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(VITOCM_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
  return 0;
}
int make_tmap_bf16(CUtensorMap* tm, const void* ptr, long long rows, long long cols, long long ld, int box_rows) {
  return make_tmap(tm, ptr, false, cols, rows, ld, 64, box_rows, CU_TENSOR_MAP_SWIZZLE_128B);
}

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  bool owned = true;   // false: caller-owned device memory (vitocm_bind_weight)
  ~DevBuf() { if (p && owned) cudaFree(p); }
  void bind(void* ptr, size_t n) {
    if (p && owned) cudaFree(p);
    p = ptr; bytes = n; owned = false;
  }
  int alloc(size_t n) {
    if (p && owned && bytes == n) return 0;   // repack in place (vitocm_refresh_weights)
    if (p && owned) cudaFree(p);
    p = nullptr; owned = true;
    bytes = n;
    cudaError_t e = cudaMalloc(&p, n ? n : 1);
    if (e != cudaSuccess) { p = nullptr; return fail(VITOCM_ERR_CUDA, "cudaMalloc(%zu) failed: %s", n, cudaGetErrorString(e)); }
    return 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct LayerW {
  DevBuf wqkv, wproj, w1, w2;      // bf16 [rows][K * parts]  (hi | lo)
  DevBuf wk_split;                 // last layer: K rows of qkv, always split [D][2D]
  // single 16-bit inference engines (vitocm_finalize_weights): W1 diag(norm2.weight), b1 + W1 norm2.bias and Wqkv diag(norm1.weight),
  // bqkv + Wqkv norm1.bias -- the block-tail kernel then skips the LayerNorm affine step (fold_ln_weight_kernel)
  DevBuf w1_fold, b1_fold, wqkv_fold, bqkv_fold;
  DevBuf wqkv_t, wproj_t, w1_t, w2_t;   // bf16 [K][rows]: transposed copies, the B operand of the input-gradient GEMMs (bf16 engines)
  const float *bqkv = nullptr, *bproj = nullptr, *b1 = nullptr, *b2 = nullptr;
  const float *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr, *ln2b = nullptr;
  const float* wqkv_f32 = nullptr;  // master copy (q rows used by the CLS kernel)
};

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
// bytes of a caller workspace [ws, ws + ws_bytes) left after aligning its start up to `base` (0 when the slack alone exceeds it)
size_t ws_avail(const void* ws, const void* base, size_t ws_bytes) {
  const size_t slack = reinterpret_cast<uintptr_t>(base) - reinterpret_cast<uintptr_t>(ws);
  return ws_bytes > slack ? ws_bytes - slack : 0;
}

}  // namespace

struct vitocm_engine {
  vitocm_config cfg{};
  int split = 0;         // fp32-parity mode: every operand a (hi, lo) pair, three MMAs per product
  int parts = 1;
  int f16 = 0;           // fp16 engines: all 16-bit tensor-core operands are IEEE half instead of bf16
  std::vector<int> layer_mode;   // per block: 0 = the engine's mode; 1 = fc1 / fc2 read their activations as (hi, lo) pairs (two MMAs
                                 // per product, single-precision weights): vitocm_set_layer_mode
  bool any_mlp_split() const { for (int m : layer_mode) if (m == 1) return true; return false; }
  int num_sms = 148;
  bool finalized = false;
  bool fold_valid = false;   // LayerW::*_fold match the master weights (set by vitocm_finalize_weights, cleared by every other weight change)
  int tail_fold = 1;         // VITOCM_TAIL_FOLD (read at vitocm_create): 0 = the block tail applies gamma / beta itself
  std::map<std::string, DevBuf*> master;  // fp32 weights as loaded
  std::vector<LayerW> layers;
  DevBuf patch_w;   // bf16 [D][2K]  (hi | lo): the conv filter as a K-major GEMM operand
  DevBuf patch_w_gray_f32, patch_w_gray;   // the filter summed over input channels, fp32 [D][p*p] and bf16 [D][2 p*p]: gray fast path
  DevBuf dec_w;     // MIM decoder 1x1 conv weight, bf16 [C p^2][D * parts] (present iff "decoder.0.weight" was loaded)
  DevBuf dec_w_t;   // bf16 [D][C p^2] (training)
  DevBuf patch_w_t;          // 16-bit [C p^2][D]: the transposed patch filter, B operand of the input-gradient GEMM
  bool patch_w_t_on = false; // set by the first vitocm_encoder_backward that asks for dx; the repack keeps patch_w_t from then on
  DevBuf repack_table;   // RepackEntry[] for the one-launch repack of the Linear weights (bf16 engines)
  int repack_entries = 0, repack_tiles = 0;
  std::vector<const void*> repack_key;   // the pointers the table was built for
  std::map<std::string, float*> grads;   // vitocm_bind_grad: where vitocm_mim_backward accumulates dL/d(parameter)
  // chunk-level concurrency: independent chunks of tiles run on `lanes` streams (lane 0 = the caller's stream) so that
  // one chunk's kernel tails and bandwidth-bound kernels overlap the other chunk's tensor-bound kernels
  static constexpr int MAX_LANES = 4;
  int lanes = 1;
  cudaStream_t aux[MAX_LANES - 1] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[MAX_LANES - 1] = {nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> bwd_events;   // vitocm_mim_backward_events: [depth] blocks + [1] head, recorded as the gradient buckets complete
  ~vitocm_engine() {
    for (cudaEvent_t ev : bwd_events) if (ev) cudaEventDestroy(ev);
    for (auto& kv : master) delete kv.second;
    for (int i = 0; i < MAX_LANES - 1; ++i) {
      if (aux[i]) cudaStreamDestroy(aux[i]);
      if (ev_join[i]) cudaEventDestroy(ev_join[i]);
    }
    if (ev_fork) cudaEventDestroy(ev_fork);
  }
  const float* w(const std::string& name) const {
    auto it = master.find(name);
    return it == master.end() ? nullptr : it->second->as<float>();
  }
  long long numel(const std::string& name) const {
    auto it = master.find(name);
    return it == master.end() ? -1 : static_cast<long long>(it->second->bytes / 4);
  }
};

namespace {

// ---------------------------------------------------------------------------------- GEMM launch
template <int BN, int EPI, bool A_PATCH>
int launch_gemm_inst(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& a, int num_sms,
                     cudaStream_t st, const CUtensorMap* td = nullptr) {
  using Cfg = GemmCfg<BN, EPI>;
  static bool attr_set = false;
  auto kern = gemm_bf16_tcgen05_kernel<BN, EPI, A_PATCH, false>;
  if (!attr_set) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int tiles = ((a.M + GEMM_BM - 1) / GEMM_BM) * (a.N / BN);
  const int grid = tiles < num_sms ? tiles : num_sms;
  kern<<<grid, gemm_threads(BN, EPI), Cfg::SMEM_BYTES, st>>>(ta, tb, tc, td ? *td : tc, a);
  LAUNCH_CHECK();
  return 0;
}

// weight-panel-resident variant (K <= 384, single-bf16 operands): see GemmCfg
template <int BN, int EPI>
int launch_gemm_res(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, GemmArgs a, int num_sms, cudaStream_t st) {
  using Cfg = GemmCfg<BN, EPI, true>;
  static int attr_bytes = 0;
  auto kern = gemm_bf16_tcgen05_kernel<BN, EPI, false, true>;
  const int smem = Cfg::res_smem_bytes(a.kblocks);
  if (smem > attr_bytes) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_bytes = smem;
  }
  a.stages = Cfg::res_stages(a.kblocks);
  const int tiles = ((a.M + GEMM_BM - 1) / GEMM_BM) * (a.N / BN);
  const int grid = tiles < num_sms ? tiles : num_sms;
  kern<<<grid, gemm_threads(BN, EPI), smem, st>>>(ta, tb, tc, tc, a);
  LAUNCH_CHECK();
  return 0;
}

// proj / fc2 with the following LayerNorm fused (EPI_RESID_LN): clusters of CS = N / BN CTAs, one per column tile
template <int BN, int CS>
int launch_gemm_ln(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& td, GemmArgs a, int num_sms,
                   cudaStream_t st) {
  using Cfg = GemmCfg<BN, EPI_RESID_LN, false, CS>;
  static int max_clusters = -1;
  auto kern = gemm_bf16_tcgen05_kernel<BN, EPI_RESID_LN, false, false, CS>;
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(gemm_threads(BN, EPI_RESID_LN));
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (max_clusters < 0) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    cfg.gridDim = dim3(CS * (num_sms / CS));
    int n = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n < 1) return fail(VITOCM_ERR_CUDA, "no %d-CTA cluster of the fused-LayerNorm GEMM fits on this device", CS);
    max_clusters = n < num_sms / CS ? n : num_sms / CS;
  }
  const int tiles_m = (a.M + GEMM_BM - 1) / GEMM_BM;
  a.num_clusters = tiles_m < max_clusters ? tiles_m : max_clusters;
  cfg.gridDim = dim3(CS * a.num_clusters);
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, td, a));
  LAUNCH_CHECK();
  return 0;
}

// cta_group::2 variant: clusters of two CTAs share 256 x BN tiles (see GemmCfg)
template <int BN, int EPI>
int launch_gemm_pair(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& a, int num_sms, cudaStream_t st,
                     const CUtensorMap* td = nullptr) {
  using Cfg = GemmCfg<BN, EPI, false, 1, true>;
  static int max_pairs = -1;
  auto kern = gemm_bf16_tcgen05_kernel<BN, EPI, false, false, 1, true>;
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(gemm_threads(BN, EPI));
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (max_pairs < 0) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    cfg.gridDim = dim3(2 * (num_sms / 2));
    int n = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n < 1) return fail(VITOCM_ERR_CUDA, "no CTA pair of the cta_group::2 GEMM fits on this device");
    max_pairs = n < num_sms / 2 ? n : num_sms / 2;
  }
  const int tiles = ((a.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM)) * (a.N / BN);
  cfg.gridDim = dim3(2 * (tiles < max_pairs ? tiles : max_pairs));
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, td ? *td : tc, a));
  LAUNCH_CHECK();
  return 0;
}

template <int BN>
int launch_gemm_pair_bn(int epi, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& a, int num_sms,
                        cudaStream_t st, const CUtensorMap* td = nullptr) {
  switch (epi) {
    case EPI_BIAS_BF16: return launch_gemm_pair<BN, EPI_BIAS_BF16>(ta, tb, tc, a, num_sms, st);
    case EPI_BIAS_GELU_BF16: return launch_gemm_pair<BN, EPI_BIAS_GELU_BF16>(ta, tb, tc, a, num_sms, st);
    case EPI_BIAS_RESID_F32: return launch_gemm_pair<BN, EPI_BIAS_RESID_F32>(ta, tb, tc, a, num_sms, st);
    case EPI_BIAS_F32: return launch_gemm_pair<BN, EPI_BIAS_F32>(ta, tb, tc, a, num_sms, st);
    case EPI_DGELU_BF16: return launch_gemm_pair<BN, EPI_DGELU_BF16>(ta, tb, tc, a, num_sms, st, td);
  }
  return fail(VITOCM_ERR_INVALID, "unknown GEMM epilogue %d", epi);
}

template <int BN>
int launch_gemm_bn(int epi, bool res, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmArgs& a,
                   int num_sms, cudaStream_t st, const CUtensorMap* td = nullptr) {
  if constexpr (BN == 192 || BN == 128) {
    if (res) {
      switch (epi) {
        case EPI_BIAS_BF16: return launch_gemm_res<BN, EPI_BIAS_BF16>(ta, tb, tc, a, num_sms, st);
        case EPI_BIAS_GELU_BF16: return launch_gemm_res<BN, EPI_BIAS_GELU_BF16>(ta, tb, tc, a, num_sms, st);
        case EPI_BIAS_RESID_F32: return launch_gemm_res<BN, EPI_BIAS_RESID_F32>(ta, tb, tc, a, num_sms, st);
        case EPI_BIAS_F32: return launch_gemm_res<BN, EPI_BIAS_F32>(ta, tb, tc, a, num_sms, st);
      }
    }
  }
  switch (epi) {
    case EPI_BIAS_BF16: return launch_gemm_inst<BN, EPI_BIAS_BF16, false>(ta, tb, tc, a, num_sms, st);
    case EPI_BIAS_GELU_BF16: return launch_gemm_inst<BN, EPI_BIAS_GELU_BF16, false>(ta, tb, tc, a, num_sms, st);
    case EPI_BIAS_RESID_F32: return launch_gemm_inst<BN, EPI_BIAS_RESID_F32, false>(ta, tb, tc, a, num_sms, st);
    case EPI_BIAS_F32: return launch_gemm_inst<BN, EPI_BIAS_F32, false>(ta, tb, tc, a, num_sms, st);
    case EPI_DGELU_BF16: return launch_gemm_inst<BN, EPI_DGELU_BF16, false>(ta, tb, tc, a, num_sms, st, td);
  }
  return fail(VITOCM_ERR_INVALID, "unknown GEMM epilogue %d", epi);
}

// Tile width: among the instantiated BN that divide N, minimise (tiles per CTA of the persistent grid) x (per-tile
// cost ~ BN + fixed overhead) -- e.g. N = 384, M = 25120 on 148 SMs: BN = 192 needs 3 rounds of 394 tiles,
// BN = 128 needs 4 rounds of 591 smaller tiles and wins.
int pick_bn(int M, int N, int num_sms, int max_bn) {
  const int cand[4] = {256, 192, 128, 64};
  const long long tiles_m = (M + GEMM_BM - 1) / GEMM_BM;
  int best = 0;
  long long best_cost = 0;
  for (int bn : cand) {
    if (bn > max_bn || N % bn != 0) continue;
    const long long tiles = tiles_m * (N / bn);
    const long long waves = (tiles + num_sms - 1) / num_sms;
    const long long cost = waves * (bn + 48);
    if (best == 0 || cost < best_cost) { best = bn; best_cost = cost; }
  }
  return best;
}

// A [M][lda] (split: hi at col 0, lo at col K), B [N][ldb] likewise.
int run_gemm(const vitocm_engine* e, const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
             int split_in, int epi, const float* bias, void* out, long long ldo, int split_out, int lo_off, cudaStream_t st,
             int pcls = PC_OTHER, const void* pre = nullptr, long long ld_pre = 0) {
  if (epi == EPI_DGELU_BF16 && (pre == nullptr || split_in || ld_pre % 8 != 0 || (reinterpret_cast<uintptr_t>(pre) & 15) != 0))
    return fail(VITOCM_ERR_INVALID, "GEMM dGELU epilogue needs a 16-byte aligned bf16 pre-activation and single-bf16 operands");
  if (M <= 0) return 0;
  ProfScope prof(pcls, st);
  if (K % GEMM_BK != 0) return fail(VITOCM_ERR_INVALID, "GEMM K=%d must be a multiple of %d", K, GEMM_BK);
  if (N % 64 != 0) return fail(VITOCM_ERR_INVALID, "GEMM N=%d must be a multiple of 64", N);
  if (bias != nullptr && (reinterpret_cast<uintptr_t>(bias) & 15) != 0) return fail(VITOCM_ERR_INVALID, "GEMM bias must be 16-byte aligned");
  // cta_group::2 (CTA pairs on 256-row tiles): single-bf16 operands, enough rows to fill the pairs
  static const int pair_mode = [] { const char* v = getenv("VITOCM_GEMM_PAIR"); return v ? atoi(v) : GEMM_PAIR_DEFAULT; }();
  // measured (profiles/r01_gemm_pair.txt): pairs win once the launch is long enough to amortise the cluster lockstep
  // (M = 137k: qkv +21 %, fc2 +6 %, fc1 +3 %) and for long K at any size; mode 2 forces pairs wherever legal
  const bool pair_pays = pair_mode == 2 || M >= 65536 || (K >= 1024 && M >= 4096);
  if (pair_mode != 0 && pair_pays && split_in != 1 && M >= 4 * GEMM_BM && (N % 256 == 0 || N % 192 == 0 || N % 128 == 0)) {
    static const int gelu_bn = [] { const char* v = getenv("VITOCM_GELU_BN"); return v ? atoi(v) : 192; }();   // measured: 835 vs 794 TFLOP/s
    int pbn = N % 256 == 0 ? 256 : (N % 192 == 0 ? 192 : 128);
    if ((epi == EPI_BIAS_GELU_BF16 || epi == EPI_DGELU_BF16) && gelu_bn == 192 && N % 192 == 0) pbn = 192;   // 12 epilogue warps instead of 8
    const bool of32 = (epi == EPI_BIAS_RESID_F32 || epi == EPI_BIAS_F32);
    CUtensorMap pa, pb, pc;
    TRY(make_tmap_bf16(&pa, A, M, split_in == 2 ? 2LL * K : K, lda, GEMM_BM));
    TRY(make_tmap_bf16(&pb, B, N, K, ldb, pbn / 2));
    TRY(make_tmap(&pc, out, of32, ldo, M, ldo, 32, 32, of32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B));
    GemmArgs pg{};
    pg.M = M; pg.N = N; pg.kblocks = K / GEMM_BK; pg.nterms = split_in == 2 ? 2 : 1; pg.lo_k = K; pg.a_lo_mask = split_in == 2 ? 2 : 0; pg.b_lo_mask = 0;
    pg.f16 = e->f16; pg.gelu_mode = e->f16 ? 2 : 0;
    pg.bias = bias; pg.out_f32 = reinterpret_cast<float*>(out);
    pg.split_out = split_out; pg.lo_off = lo_off;
    pg.pre = reinterpret_cast<const __nv_bfloat16*>(pre); pg.ld_pre = ld_pre;
    CUtensorMap pd;
    const CUtensorMap* ppd = nullptr;
    if (epi == EPI_DGELU_BF16) {   // the saved pre-activation, read by the epilogue as 32 x 32 bf16 boxes
      TRY(make_tmap(&pd, pre, false, N, M, ld_pre, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B));
      ppd = &pd;
    }
    { static const int dbgp = [] { const char* v = getenv("VITOCM_GEMM_DEBUG"); return v ? atoi(v) : 0; }(); pg.debug = dbgp; }
    if (pbn == 256) return launch_gemm_pair_bn<256>(epi, pa, pb, pc, pg, e->num_sms, st, ppd);
    if (pbn == 192) return launch_gemm_pair_bn<192>(epi, pa, pb, pc, pg, e->num_sms, st, ppd);
    return launch_gemm_pair_bn<128>(epi, pa, pb, pc, pg, e->num_sms, st, ppd);
  }
  static const bool allow_res = [] { const char* v = getenv("VITOCM_GEMM_RESIDENT"); return v == nullptr || atoi(v) != 0; }();
  // weight panel resident in smem: single-bf16 operands, K <= 384, tile width 192 or 128
  bool res = allow_res && !split_in && !split_out && epi != EPI_DGELU_BF16 && K / GEMM_BK <= GEMM_RES_MAX_KBLOCKS && (N % 128 == 0 || N % 192 == 0);
  const int bn = pick_bn(M, N, e->num_sms, res ? 192 : 256);
  if (res && bn < 128) res = false;
  const long long kext = static_cast<long long>(K) * (split_in ? 2 : 1);
  const bool out_f32 = (epi == EPI_BIAS_RESID_F32 || epi == EPI_BIAS_F32);
  CUtensorMap ta, tb, tc;
  TRY(make_tmap_bf16(&ta, A, M, kext, lda, GEMM_BM));
  TRY(make_tmap_bf16(&tb, B, N, split_in == 2 ? K : kext, ldb, bn));
  TRY(make_tmap(&tc, out, out_f32, ldo, M, ldo, 32, 32, out_f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B));
  GemmArgs a{};
  // split_in: 0 = single operands (1 MMA per product); 1 = A and B as (hi, lo) pairs, hi*hi + hi*lo + lo*hi; 2 = A as a pair, B single
  a.M = M; a.N = N; a.kblocks = K / GEMM_BK; a.nterms = split_in == 1 ? 3 : (split_in == 2 ? 2 : 1);
  a.a_lo_mask = split_in == 1 ? 4 : (split_in == 2 ? 2 : 0); a.b_lo_mask = split_in == 1 ? 2 : 0;
  a.f16 = e->f16; a.gelu_mode = split_in == 1 ? 1 : (e->f16 ? 2 : 0);
  a.lo_k = K;
  a.bias = bias; a.split_out = split_out; a.lo_off = lo_off;
  static const int dbg = [] { const char* v = getenv("VITOCM_GEMM_DEBUG"); return v ? atoi(v) : 0; }();
  a.debug = dbg; a.out_f32 = reinterpret_cast<float*>(out);
  a.pre = reinterpret_cast<const __nv_bfloat16*>(pre); a.ld_pre = ld_pre;
  CUtensorMap td;
  const CUtensorMap* ptd = nullptr;
  if (epi == EPI_DGELU_BF16) {
    TRY(make_tmap(&td, pre, false, N, M, ld_pre, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B));
    ptd = &td;
  }
  switch (bn) {
    case 256: return launch_gemm_bn<256>(epi, res, ta, tb, tc, a, e->num_sms, st, ptd);
    case 192: return launch_gemm_bn<192>(epi, res, ta, tb, tc, a, e->num_sms, st, ptd);
    case 128: return launch_gemm_bn<128>(epi, res, ta, tb, tc, a, e->num_sms, st, ptd);
    default: return launch_gemm_bn<64>(epi, res, ta, tb, tc, a, e->num_sms, st, ptd);
  }
}

// X[M][N] += A . B^T + bias;  XN = bf16(LayerNorm(X) * gamma + beta)   (single-bf16 operands only).
// Returns 1 when the shape has no fused instantiation (the caller then runs the two kernels separately).
int run_gemm_ln(const vitocm_engine* e, const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
                const float* bias, float* X, const float* gamma, const float* beta, float eps, void* XN, long long ld_xn,
                cudaStream_t st, int pcls) {
  // VITOCM_FUSE_LN: 0 = never, 1 = short-K GEMMs only (proj; default -- measured: the long-K fc2 is L2-bandwidth bound and
  // loses more to the extra residual traffic and the per-tile cluster lockstep than the LayerNorm kernel costs), 2 = always
  static const int mode = [] { const char* v = getenv("VITOCM_FUSE_LN"); return v == nullptr ? 1 : atoi(v); }();
  if (mode == 0 || (mode == 1 && K > 512 && pcls != PC_OTHER)) return 1;
  if (e->split || M <= 0 || K % GEMM_BK != 0 || bias == nullptr) return 1;
  // one cluster of CS = N / 128 CTAs spans a row (cluster sizes 1, 2, 3, 4, 6: N = 128 ... 768)
  if (N % 128 != 0) return 1;
  const int cs = N / 128;
  if (cs != 1 && cs != 2 && cs != 3 && cs != 4 && cs != 6) return 1;
  ProfScope prof(pcls, st);
  CUtensorMap ta, tb, tc, td;
  TRY(make_tmap_bf16(&ta, A, M, K, lda, GEMM_BM));
  TRY(make_tmap_bf16(&tb, B, N, K, ldb, 128));
  TRY(make_tmap(&tc, X, true, N, M, N, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B));
  TRY(make_tmap(&td, XN, false, ld_xn, M, ld_xn, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B));
  GemmArgs a{};
  a.M = M; a.N = N; a.kblocks = K / GEMM_BK; a.nterms = 1; a.lo_k = K; a.f16 = e->f16;
  a.bias = bias; a.out_f32 = X;
  a.ln_gamma = gamma; a.ln_beta = beta; a.ln_eps = eps;
  a.xn = reinterpret_cast<__nv_bfloat16*>(XN); a.ld_xn = ld_xn;
  switch (cs) {
    case 1: return launch_gemm_ln<128, 1>(ta, tb, tc, td, a, e->num_sms, st);
    case 2: return launch_gemm_ln<128, 2>(ta, tb, tc, td, a, e->num_sms, st);
    case 3: return launch_gemm_ln<128, 3>(ta, tb, tc, td, a, e->num_sms, st);
    case 4: return launch_gemm_ln<128, 4>(ta, tb, tc, td, a, e->num_sms, st);
    default: return launch_gemm_ln<128, 6>(ta, tb, tc, td, a, e->num_sms, st);
  }
}

// ---------------------------------------------------------------------------------- fused MLP launch
// X[M][D] += gelu(XN . W1^T + b1) . W2^T + b2 in one kernel (mlp_fused_sm100.cuh).  Returns 1 when the shape / engine has no
// fused instantiation (the caller then runs fc1 and fc2 as separate GEMMs).
template <int KB1, int CL>
int launch_mlp_fused(const CUtensorMap& ta, const CUtensorMap& tw1, const CUtensorMap& tw2, const CUtensorMap& tx, MlpArgs a,
                     int num_sms, cudaStream_t st) {
  using Cfg = MlpCfg<KB1, CL>;
  static int max_clusters = -1;
  auto kern = mlp_fused_tcgen05_kernel<KB1, CL>;
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (max_clusters < 0) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    if (CL > 2) CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cfg.gridDim = dim3(CL * (num_sms / CL));
    int n = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n < 1) return fail(VITOCM_ERR_CUDA, "no %d-CTA cluster of the fused MLP kernel fits on this device", CL);
    max_clusters = n < num_sms / CL ? n : num_sms / CL;
  }
  const int tiles = (a.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM);
  const int groups = (tiles + CL / 2 - 1) / (CL / 2);
  const int nclusters = groups < max_clusters ? groups : max_clusters;
  // clusters [groups % nclusters, nclusters) have one work item fewer than the others: they start late, spread over one item's time
  static const int stagger = [] { const char* v = getenv("VITOCM_MLP_STAGGER"); return v ? atoi(v) : 40000; }();
  a.stagger_from = (stagger > 0 && groups > nclusters && groups % nclusters != 0) ? groups % nclusters : nclusters;
  a.stagger_clk = stagger;
  cfg.gridDim = dim3(CL * nclusters);
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ta, tw1, tw2, tx, a));
  LAUNCH_CHECK();
  return 0;
}

int run_mlp_fused(const vitocm_engine* e, const void* XN, long long ld_xn, const void* W1, long long ldw1, const void* W2, long long ldw2,
                  int M, int D, int Hd, const float* b1, const float* b2, float* X, cudaStream_t st, bool force = false,
                  long long* timeline = nullptr) {
  // VITOCM_FUSE_MLP: 0 = never (fc1 and fc2 as separate GEMMs), otherwise the cluster size: 2 (default: one CTA pair per cluster) or
  // 4 (two pairs share every weight tile through TMA multicast: half the L2 -> SM weight traffic, but measured 5 % SLOWER -- the
  // kernel is bound by the GELU arithmetic and by shared-memory reads of its N = 128 MMAs, not by the weight stream, and four
  // CTAs in lockstep lose more than the traffic saves; profiles/r02_mlp_fused.txt)
  static const int mode = [] { const char* v = getenv("VITOCM_FUSE_MLP"); return v == nullptr ? 2 : atoi(v); }();
  if (mode == 0 && !force) return 1;
  if (e->split || M <= 0 || (D != 128 && D != 384) || Hd % MLP_HC != 0 || b1 == nullptr || b2 == nullptr) return 1;
  if ((reinterpret_cast<uintptr_t>(b1) & 15) != 0 || (reinterpret_cast<uintptr_t>(b2) & 15) != 0) return 1;
  ProfScope prof(PC_MLP, st);
  CUtensorMap ta, tw1, tw2, tx;
  TRY(make_tmap_bf16(&ta, XN, M, D, ld_xn, GEMM_BM));
  TRY(make_tmap_bf16(&tw1, W1, Hd, D, ldw1, 64));
  TRY(make_tmap_bf16(&tw2, W2, D, Hd, ldw2, D == 384 ? 96 : 64));   // one CTA's half of a [BN2 x 64] tile: BN2 = 192 at D = 384
  TRY(make_tmap(&tx, X, true, D, M, D, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B));   // output staging boxes: 32 rows x 32 fp32 columns
  MlpArgs a{};
  a.M = M; a.hidden = Hd; a.f16 = e->f16; a.gelu_mode = e->f16 ? 2 : 0; a.bias1 = b1; a.bias2 = b2;
  a.timeline = timeline;
  { static const int dbg = [] { const char* v = getenv("VITOCM_MLP_DEBUG"); return v ? atoi(v) : 0; }(); a.debug = dbg; }
  { static const int tli = [] { const char* v = getenv("VITOCM_MLP_TL_ITEM"); return v ? atoi(v) : 1; }(); a.timeline_item = tli; }
  const bool pair_only = mode != 4;
  if (D == 384) return pair_only ? launch_mlp_fused<6, 2>(ta, tw1, tw2, tx, a, e->num_sms, st) : launch_mlp_fused<6, 4>(ta, tw1, tw2, tx, a, e->num_sms, st);
  return pair_only ? launch_mlp_fused<2, 2>(ta, tw1, tw2, tx, a, e->num_sms, st) : launch_mlp_fused<2, 4>(ta, tw1, tw2, tx, a, e->num_sms, st);
}

// ---------------------------------------------------------------------------------- block tail launch
// proj + residual + norm2 + fc1 + GELU + fc2 + residual (+ the next LayerNorm) in one kernel (block_tail_sm100.cuh).  Returns 1 when
// the shape / engine has no instantiation (the caller then runs the separate kernels).
template <int KB1, bool F16>
int launch_block_tail(const CUtensorMap& ta, const CUtensorMap& twp, const CUtensorMap& tw1, const CUtensorMap& tw2, const CUtensorMap& tx,
                      const CUtensorMap& txn, const CUtensorMap& twqkv, const CUtensorMap& tqkv, const TailArgs& a, int num_sms, cudaStream_t st) {
  using Cfg = TailCfg<KB1>;
  static int max_clusters = -1;
  auto kern = block_tail_tcgen05_kernel<KB1, F16>;
  cudaLaunchConfig_t cfg{};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (max_clusters < 0) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    cfg.gridDim = dim3(2 * (num_sms / 2));
    int n = 0;
    CUDA_TRY(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    if (n < 1) return fail(VITOCM_ERR_CUDA, "no CTA pair of the block-tail kernel fits on this device");
    max_clusters = n < num_sms / 2 ? n : num_sms / 2;
  }
  const int tiles = (a.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM);
  cfg.gridDim = dim3(2 * (tiles < max_clusters ? tiles : max_clusters));
  CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ta, twp, tw1, tw2, tx, txn, twqkv, tqkv, a));
  LAUNCH_CHECK();
  return 0;
}

// Wqkv != nullptr (needs lnn_w): the kernel also computes the NEXT block's QKV = LayerNorm(X; lnn) . Wqkv^T + bqkv into QKV [M][ld_qkv]
// and XN is not written.
int run_block_tail(const vitocm_engine* e, const void* CTX, long long ld_ctx, const void* Wp, long long ldwp, const float* bp,
                   const float* ln2w, const float* ln2b, const void* W1, long long ldw1, const void* W2, long long ldw2, int M, int D, int Hd,
                   const float* b1, const float* b2, float* X, const float* lnn_w, const float* lnn_b, float eps, void* XN, long long ld_xn,
                   const void* Wqkv, long long ldwqkv, const float* bqkv, void* QKV, long long ld_qkv,
                   cudaStream_t st, bool force = false, long long* timeline = nullptr, bool fold2 = false, bool foldn = false) {
  // fold2: W1 / b1 carry norm2's gamma / beta; foldn: Wqkv / bqkv carry the next norm1's (LayerW::*_fold; with Wqkv only)
  // VITOCM_FUSE_TAIL: 0 = never (proj + LayerNorm GEMM, fused MLP and LayerNorm as separate kernels), 1 = default
  static const int mode = [] { const char* v = getenv("VITOCM_FUSE_TAIL"); return v == nullptr ? 1 : atoi(v); }();
  if (mode == 0 && !force) return 1;
  if (e->split || M <= 0 || (D != 128 && D != 384) || Hd % MLP_HC != 0) return 1;
  const float* vecs[8] = {bp, ln2w, ln2b, b1, b2, lnn_w, lnn_b, bqkv};
  for (int i = 0; i < 8; ++i) {
    if (i < 5 && vecs[i] == nullptr) return 1;
    if ((reinterpret_cast<uintptr_t>(vecs[i]) & 15) != 0) return 1;
  }
  if ((lnn_w == nullptr) != (lnn_b == nullptr)) return 1;
  const bool with_qkv = Wqkv != nullptr;
  if (with_qkv && (lnn_w == nullptr || bqkv == nullptr || QKV == nullptr)) return 1;
  if (!with_qkv && lnn_w != nullptr && XN == nullptr) return 1;
  ProfScope prof(PC_TAIL, st);
  CUtensorMap ta, twp, tw1, tw2, tx, txn, twqkv, tqkv;
  const int w2_rows = D == 384 ? 96 : 64;   // one CTA's half of a [BN2 x 64] tile: BN2 = 192 at D = 384
  TRY(make_tmap_bf16(&ta, CTX, M, D, ld_ctx, GEMM_BM));
  TRY(make_tmap_bf16(&twp, Wp, D, D, ldwp, w2_rows));
  TRY(make_tmap_bf16(&tw1, W1, Hd, D, ldw1, 64));
  TRY(make_tmap_bf16(&tw2, W2, D, Hd, ldw2, w2_rows));
  TRY(make_tmap(&tx, X, true, D, M, D, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B));
  if (lnn_w != nullptr && !with_qkv) TRY(make_tmap(&txn, XN, false, ld_xn, M, ld_xn, 32, 32, CU_TENSOR_MAP_SWIZZLE_64B));
  else txn = tx;
  if (with_qkv) {
    TRY(make_tmap_bf16(&twqkv, Wqkv, 3LL * D, D, ldwqkv, 64));
    TRY(make_tmap_bf16(&tqkv, QKV, M, 3LL * D, ld_qkv, 32));   // one warp's 32 rows x 64 columns per store
  } else {
    twqkv = tw1; tqkv = ta;
  }
  TailArgs a{};
  a.M = M; a.hidden = Hd; a.gelu5 = e->f16 ? 1 : 0;
  a.bias_p = bp; a.ln2_w = ln2w; a.ln2_b = ln2b; a.bias1 = b1; a.bias2 = b2; a.lnn_w = lnn_w; a.lnn_b = lnn_b; a.ln_eps = eps;
  a.bias_qkv = bqkv; a.n_qkv_chunks = with_qkv ? 3 * D / MLP_HC : 0;
  a.fold2 = fold2 ? 1 : 0; a.foldn = (foldn && with_qkv) ? 1 : 0;
  a.timeline = timeline;
  { static const int dbg = [] { const char* v = getenv("VITOCM_TAIL_DEBUG"); return v ? atoi(v) : 0; }(); a.debug = dbg; }
  {
    // Start stagger of the CTA pairs (TailArgs::stagger_clk): about one item's duration spread over the pairs, so that they sit at
    // evenly distributed phases of an item instead of all reaching the item boundary together -- 3 494 -> 3 290 us per 1 225-tile
    // launch, 538 -> 498 us per 175 tiles (profiles/r02_gpu_call_ba_tail_stagger.log).  What it costs: pair k starts k / pairs of an
    // item late; with items = n pairs + r the first r pairs carry n + 1 items, so the launch ends (r - 1) / pairs of an item later
    // (a whole item when r = 0).  The stagger is used while that stays below 4 % of the launch (the gain is 6 - 10 %); shorter
    // launches run without it.  VITOCM_TAIL_STAGGER=<clocks> overrides (0: none).
    static const int stg = [] { const char* v = getenv("VITOCM_TAIL_STAGGER"); return v ? atoi(v) : -1; }();
    if (stg >= 0) {
      a.stagger_clk = stg;
    } else {
      const long long items = (static_cast<long long>(M) + 2 * GEMM_BM - 1) / (2 * GEMM_BM);
      const long long pairs = e->num_sms / 2;
      const long long r = items % pairs, rounds = (items + pairs - 1) / pairs;
      const double late = (r > 0 ? static_cast<double>(r - 1) : static_cast<double>(pairs - 1)) / static_cast<double>(pairs);   // in items
      const double work = static_cast<double>(D) * (D + 2.0 * Hd + (with_qkv ? 3.0 * D : 0.0));   // per row, relative to ViT-S with QKV: ~105 k clk per item
      a.stagger_clk = (items > pairs && late <= 0.04 * static_cast<double>(rounds)) ? static_cast<int>(105000.0 * work / (384.0 * (384.0 + 3072.0 + 1152.0))) : 0;
    }
  }
  { static const int tli = [] { const char* v = getenv("VITOCM_MLP_TL_ITEM"); return v ? atoi(v) : 1; }(); a.timeline_item = tli; }
  if (D == 384) return e->f16 ? launch_block_tail<6, true>(ta, twp, tw1, tw2, tx, txn, twqkv, tqkv, a, e->num_sms, st) : launch_block_tail<6, false>(ta, twp, tw1, tw2, tx, txn, twqkv, tqkv, a, e->num_sms, st);
  return e->f16 ? launch_block_tail<2, true>(ta, twp, tw1, tw2, tx, txn, twqkv, tqkv, a, e->num_sms, st) : launch_block_tail<2, false>(ta, twp, tw1, tw2, tx, txn, twqkv, tqkv, a, e->num_sms, st);
}

// ---------------------------------------------------------------------------------- attention launch
int run_attention(const vitocm_engine* e, const void* qkv, long long ld, int B, int N, void* ctx, long long ldo, cudaStream_t st,
                  long long* timeline = nullptr, float* lse2 = nullptr) {
  const int D = e->cfg.embed_dim, H = e->cfg.num_heads;
  const bool hd128 = D == 128 * H;   // head_dim 128: the generic kernel's DH = 128 instantiations (no four-pipeline kernel)
  const long long M = static_cast<long long>(B) * N;
  ProfScope prof(PC_ATTN, st);
  CUtensorMap tq, tq32;
  TRY(make_tmap_bf16(&tq, qkv, M, 3LL * D * e->parts, ld, 128));
  TRY(make_tmap_bf16(&tq32, qkv, M, 3LL * D * e->parts, ld, 32));   // 32-row boxes: the query slots of packed tail items
  AttnArgs a{};
  a.n_tokens = N; a.embed_dim = D; a.lo_col_off = 3 * D;
  a.scale_log2 = e->cfg.qk_scale * 1.44269504088896340736f;
  a.out = reinterpret_cast<__nv_bfloat16*>(ctx); a.ldo = ldo; a.out_lo_off = D; a.timeline = timeline; a.lse2 = lse2;
  { static const int tli = [] { const char* v = getenv("VITOCM_ATTN_TL_ITEM"); return v ? atoi(v) : 0; }(); a.timeline_item = tli; }
  { static const int tm = [] { const char* v = getenv("VITOCM_ATTN_TRACK_MAX"); return v ? atoi(v) : 0; }(); a.track_max = tm; }
  a.n_qtiles = (N + ATT_BQ - 1) / ATT_BQ; a.heads = H;
  // ragged query tail: <= 32 rows -> 4 (image, head) pairs share one tile, <= 64 rows -> 2 (VITOCM_ATTN_PACK=0: never)
  static const int pack_on = [] { const char* v = getenv("VITOCM_ATTN_PACK"); return v ? atoi(v) : 1; }();
  const int tail = N % ATT_BQ;
  a.n_fullq = N / ATT_BQ;
  // (only where the tail tiles are a visible share of the work: beyond 16 full tiles per pair the slot logic costs more than it saves)
  a.pack = (!pack_on || tail == 0 || tail > 64 || a.n_fullq > 16) ? 1 : (tail > 32 ? 2 : 4);
  a.group_items = a.pack * a.n_fullq + (tail != 0 ? 1 : 0);
  a.n_pairs = B * H;
  const long long items = static_cast<long long>((a.n_pairs + a.pack - 1) / a.pack) * a.group_items;
  if (items > 0x7fffffffLL) return fail(VITOCM_ERR_INVALID, "attention: too many work items");
  a.n_items = static_cast<int>(items);
  // 16-bit engines, inference: the full query tiles go through the four-pipeline kernel (attention_quad_sm100.cuh), the ragged
  // tails through the packed items of the kernel below (VITOCM_ATTN_QUAD=0: everything through the kernel below)
  static const int quad = [] { const char* v = getenv("VITOCM_ATTN_QUAD"); return v ? atoi(v) : 1; }();
  if (quad && !hd128 && !e->split && lse2 == nullptr && a.n_fullq >= 1) {
    const long long full_items = static_cast<long long>(a.n_pairs) * a.n_fullq;
    if (full_items > 0x7fffffffLL) return fail(VITOCM_ERR_INVALID, "attention: too many work items");
    AttnArgs aq = a;
    aq.n_full_items = static_cast<int>(full_items);
    // the ragged query tails ride along as the kernel's last items when they pack (a.pack > 1: `pack` pairs per tile); otherwise
    // (VITOCM_ATTN_QUAD_TAILS=0, a tail of more than 64 rows, more than 16 full tiles per pair) they go through the kernel below
    static const int quad_tails = [] { const char* v = getenv("VITOCM_ATTN_QUAD_TAILS"); return v ? atoi(v) : 1; }();
    const bool tails_here = quad_tails && a.pack > 1;
    static const int quad_pack = [] { const char* v = getenv("VITOCM_ATTN_QUAD_PACK"); return v ? atoi(v) : 2; }();   // 2 or 4
    aq.group_items = 0;
    { static const int hoist = [] { const char* v = getenv("VITOCM_ATTN_HOIST"); return v ? atoi(v) : 1; }(); aq.ctrl_hoist = hoist; }
    { static const int stg = [] { const char* v = getenv("VITOCM_ATTN_STAGGER"); return v ? atoi(v) : 0; }(); aq.stagger_clk = stg; }
    aq.n_items = aq.n_full_items;
    if (tails_here) {   // groups of `pack` pairs: their full tiles, then the one tile their tails share (aq_decode)
      aq.pack = (quad_pack == 4 && a.pack == 4) ? 4 : 2;
      aq.group_items = aq.pack * a.n_fullq + 1;
      const long long gi = static_cast<long long>((a.n_pairs + aq.pack - 1) / aq.pack) * aq.group_items;
      if (gi > 0x7fffffffLL) return fail(VITOCM_ERR_INVALID, "attention: too many work items");
      aq.n_items = static_cast<int>(gi);
    }
    CUtensorMap tkv;
    TRY(make_tmap_bf16(&tkv, qkv, M, 3LL * D * e->parts, ld, AQ_BKV));
    const int ctas = (aq.n_items + AQ_PIPES - 1) / AQ_PIPES;
    const dim3 qgrid(ctas < e->num_sms ? ctas : e->num_sms);
    auto qlaunch = [&](auto kern, bool& attr) -> int {
      if (!attr) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, AQ_SMEM_BYTES)); attr = true; }
      kern<<<qgrid, AQ_THREADS, AQ_SMEM_BYTES, st>>>(tq, tkv, tq32, aq);
      return 0;
    };
    static bool qattr[4] = {false, false, false, false};
    int qrc;
    if (timeline != nullptr) qrc = e->f16 ? qlaunch(attn_fwd_quad_kernel<true, true>, qattr[3]) : qlaunch(attn_fwd_quad_kernel<false, true>, qattr[2]);
    else qrc = e->f16 ? qlaunch(attn_fwd_quad_kernel<true, false>, qattr[1]) : qlaunch(attn_fwd_quad_kernel<false, false>, qattr[0]);
    if (qrc) return qrc;
    LAUNCH_CHECK();
    if (tail == 0 || tails_here) return 0;
    a.tails_only = 1;
    a.timeline = nullptr;   // (the stamps of a timeline call come from the four-pipeline kernel)
    a.n_items = (a.n_pairs + a.pack - 1) / a.pack;
  }
  // persistent CTAs: as many as are co-resident (2 per SM in bf16 mode at head_dim 64, 1 in split mode or at head_dim 128)
  const int resident = e->num_sms * ((e->split || hd128) ? 1 : 2);
  static const int persist = [] { const char* v = getenv("VITOCM_ATTN_PERSISTENT"); return v ? atoi(v) : 1; }();
  const dim3 grid(persist && a.n_items > resident ? resident : a.n_items);
  auto launch = [&](auto kern, int smem_bytes, bool& attr) -> int {
    if (!attr) { CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes)); attr = true; }
    kern<<<grid, ATT_THREADS, smem_bytes, st>>>(tq, tq32, a);
    return 0;
  };
  // (the FMA-pipe exp2 polynomial variants of round 1 measured 15-19 % slower and are no longer instantiated)
  if (hd128) {
    static bool attr128[8] = {false, false, false, false, false, false, false, false};
    if (a.pack > 1) {
      if (e->split) {
        if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, true, true, 128>, AttnCfg<true, 128>::SMEM_BYTES, attr128[1]));
        else TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, true, false, 128>, AttnCfg<true, 128>::SMEM_BYTES, attr128[3]));
      } else if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, true, true, 128>, AttnCfg<false, 128>::SMEM_BYTES, attr128[2]));
      else TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, true, false, 128>, AttnCfg<false, 128>::SMEM_BYTES, attr128[0]));
    } else {
      if (e->split) {
        if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, false, true, 128>, AttnCfg<true, 128>::SMEM_BYTES, attr128[5]));
        else TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, false, false, 128>, AttnCfg<true, 128>::SMEM_BYTES, attr128[7]));
      } else if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, false, true, 128>, AttnCfg<false, 128>::SMEM_BYTES, attr128[6]));
      else TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, false, false, 128>, AttnCfg<false, 128>::SMEM_BYTES, attr128[4]));
    }
    LAUNCH_CHECK();
    return 0;
  }
  static bool attr[8] = {false, false, false, false, false, false, false, false};
  if (a.pack > 1) {   // kernels with the packed-item logic
    if (e->split) {
      if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, true, true>, AttnCfg<true>::SMEM_BYTES, attr[1]));
      else TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, true, false>, AttnCfg<true>::SMEM_BYTES, attr[3]));
    } else if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, true, true>, AttnCfg<false>::SMEM_BYTES, attr[2]));
    else TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, true, false>, AttnCfg<false>::SMEM_BYTES, attr[0]));
  } else {
    if (e->split) {
      if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, false, true>, AttnCfg<true>::SMEM_BYTES, attr[5]));
      else TRY(launch(attn_fwd_tcgen05_kernel<true, 0u, false, false>, AttnCfg<true>::SMEM_BYTES, attr[7]));
    } else if (e->f16) TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, false, true>, AttnCfg<false>::SMEM_BYTES, attr[6]));
    else TRY(launch(attn_fwd_tcgen05_kernel<false, 0u, false, false>, AttnCfg<false>::SMEM_BYTES, attr[4]));
  }
  LAUNCH_CHECK();
  return 0;
}

int run_layernorm(const float* X, const float* g, const float* b, void* out_bf16, long long ldo, int split, int lo_off,
                  float* out_f32, long long ldf, int M, int D, float eps, cudaStream_t st, float* x_copy = nullptr, int f16 = 0) {
  if (M <= 0) return 0;
  if (D % 4 != 0 || D > LN_MAX_VEC * 128) return fail(VITOCM_ERR_INVALID, "LayerNorm D=%d unsupported", D);
  ProfScope prof(PC_LN, st);
  const int rows_per_block = 8;
  const dim3 grid((M + rows_per_block - 1) / rows_per_block), block(rows_per_block * 32);
  __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(out_bf16);
  if (D == 384) layernorm_kernel<3><<<grid, block, 0, st>>>(X, g, b, ob, ldo, split, lo_off, out_f32, ldf, M, D, eps, x_copy, f16);
  else if (D == 768) layernorm_kernel<6><<<grid, block, 0, st>>>(X, g, b, ob, ldo, split, lo_off, out_f32, ldf, M, D, eps, x_copy, f16);
  else if (D == 128) layernorm_kernel<1><<<grid, block, 0, st>>>(X, g, b, ob, ldo, split, lo_off, out_f32, ldf, M, D, eps, x_copy, f16);
  else layernorm_kernel<0><<<grid, block, 0, st>>>(X, g, b, ob, ldo, split, lo_off, out_f32, ldf, M, D, eps, x_copy, f16);
  LAUNCH_CHECK();
  return 0;
}

// prepare_tokens (vit.py:198-209) as an im2col-free tcgen05 GEMM: M = B * n patches, K = C p^2, N = D.
// tiles cut straight out of a gray uint8 mosaic by the patch-embedding producer (GemmArgs::mos)
struct MosaicSrc {
  const uint8_t* p;
  long long pitch;
  int h, w, nx, S, t0;   // nx: windows per grid row (window t has origin ((t / nx) S, (t % nx) S))
};

int run_patch_embed(const vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask,
                    float* X, cudaStream_t st, bool gray = false, const MosaicSrc* mos = nullptr) {
  // gray: x is [B][1][H][W], standing for an image with equal channels; the channel-folded filter does the same arithmetic
  const int p = e->cfg.patch_size, C = gray ? 1 : e->cfg.in_chans, D = e->cfg.embed_dim;
  if (gray && e->patch_w_gray.p == nullptr) return fail(VITOCM_ERR_STATE, "gray fast path needs in_chans > 1");
  if (H % p != 0 || W % p != 0) return fail(VITOCM_ERR_INVALID, "image %dx%d not a multiple of patch %d", H, W, p);
  const int K = C * p * p;
  if (p % 8 != 0 || K % GEMM_BK != 0) return fail(VITOCM_ERR_INVALID, "patch embedding needs patch %% 8 == 0 and C*p*p %% 64 == 0 (patch %d, chans %d)", p, C);
  if ((mos == nullptr && (reinterpret_cast<uintptr_t>(x) & 15) != 0) || (reinterpret_cast<uintptr_t>(pos) & 15) != 0)
    return fail(VITOCM_ERR_INVALID, "patch embedding inputs must be 16-byte aligned");
  if (mos != nullptr && (!gray || mos->p == nullptr || mos->nx < 1 || mos->S < 1))
    return fail(VITOCM_ERR_INVALID, "mosaic ingest needs the gray path and a valid window grid");
  const float* mask_token = e->w("mask_token");
  if (mask != nullptr && mask_token == nullptr) return fail(VITOCM_ERR_STATE, "mask given but mask_token was never loaded");
  const int n = (H / p) * (W / p);
  const int M = B * n;
  ProfScope prof(PC_PATCH, st);
  cls_rows_kernel<<<(B * D + 255) / 256, 256, 0, st>>>(e->w("cls_token"), pos, X, B, static_cast<long long>(n + 1) * D, D);
  LAUNCH_CHECK();
  const int bn = (D % 192 == 0) ? 192 : (D % 128 == 0 ? 128 : 64);
  CUtensorMap tb;
  TRY(make_tmap_bf16(&tb, gray ? e->patch_w_gray.p : e->patch_w.p, D, 2LL * K, 2LL * K, bn));
  GemmArgs a{};
  a.M = M; a.N = D; a.kblocks = K / GEMM_BK; a.nterms = 3; a.lo_k = K; a.a_lo_mask = 4; a.b_lo_mask = 2; a.f16 = e->f16;   // split precision in all modes
  a.bias = e->w("patch_embed.proj.bias");
  a.img = x; a.img_h = H; a.img_w = W; a.patch = p; a.n_patches = n; a.pos = pos; a.mask = mask; a.mask_token = mask_token; a.out_f32 = X;
  if (mos != nullptr) { a.mos = mos->p; a.mos_pitch = mos->pitch; a.mos_h = mos->h; a.mos_w = mos->w; a.mos_nx = mos->nx; a.mos_S = mos->S; a.mos_t0 = mos->t0; }
  // position rows in / token rows out through TMA boxes (VITOCM_PATCH_TMA=0: every lane reads and writes its own 128 bytes)
  static const int patch_tma = [] { const char* v = getenv("VITOCM_PATCH_TMA"); return v == nullptr ? 1 : atoi(v); }();
  CUtensorMap tx = tb, tp = tb;
  if (patch_tma && D % 32 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
    TRY(make_tmap(&tx, X, true, D, static_cast<long long>(B) * (n + 1), D, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B));
    TRY(make_tmap(&tp, pos, true, D, n + 1, D, 32, 32, CU_TENSOR_MAP_SWIZZLE_128B));
    a.patch_tma = 1;
  }
  switch (bn) {
    case 192: return launch_gemm_inst<192, EPI_PATCH_F32, true>(tb, tb, tx, a, e->num_sms, st, &tp);
    case 128: return launch_gemm_inst<128, EPI_PATCH_F32, true>(tb, tb, tx, a, e->num_sms, st, &tp);
    default: return launch_gemm_inst<64, EPI_PATCH_F32, true>(tb, tb, tx, a, e->num_sms, st, &tp);
  }
}

// workspace carve-up for a chunk of `tiles` images
struct Workspace {
  float* X;            // [M][D] fp32 token stream
  __nv_bfloat16* XN;   // [M][2D]  (always room for hi|lo: the last block's K projection is split)
  __nv_bfloat16* QKV;  // [M][3D*parts]
  __nv_bfloat16* CTX;  // [M][D*parts]
  __nv_bfloat16* HID;  // [M][4D*parts]  (aliased by KF fp32 [M][D] in the last block)
  size_t total;
};
Workspace carve(const vitocm_engine* e, void* base, int tiles, int N) {
  const size_t M = static_cast<size_t>(tiles) * N;
  const size_t D = e->cfg.embed_dim, Hd = e->cfg.mlp_hidden, P = e->parts;
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  Workspace w{};
  auto take = [&](size_t bytes) { uint8_t* r = p + off; off += align_up(bytes, 1024); return r; };
  w.X = reinterpret_cast<float*>(take(M * D * 4));
  w.XN = reinterpret_cast<__nv_bfloat16*>(take(M * 2 * D * 2));
  w.QKV = reinterpret_cast<__nv_bfloat16*>(take(M * 3 * D * P * 2));
  w.CTX = reinterpret_cast<__nv_bfloat16*>(take(M * D * P * 2));
  size_t hid = M * Hd * (e->any_mlp_split() ? 2 : P) * 2;
  if (hid < M * D * 4) hid = M * D * 4;
  w.HID = reinterpret_cast<__nv_bfloat16*>(take(hid));
  w.total = off;
  return w;
}

// one full transformer block in place on ws.X (vit.py:106-114).
// xn_ready: ws.XN already holds norm1(X) of this block (produced by the previous block's fused fc2 epilogue).
// next_ln (or null): LayerNorm parameters of the NEXT consumer of X; when the fused epilogue is available, fc2 also
// leaves that norm's output in ws.XN and *xn_done is set.
// qkv_ready: ws.QKV already holds this block's QKV projection (produced by the previous block's tail kernel); next_qkv (or null): the
// NEXT block, whose QKV projection this block's tail kernel computes when it can (*qkv_done).
int block_forward(const vitocm_engine* e, int l, const Workspace& ws, int B, int N, cudaStream_t st, bool xn_ready = false,
                  const float* next_ln_w = nullptr, const float* next_ln_b = nullptr, bool* xn_done = nullptr, bool qkv_ready = false,
                  const LayerW* next_qkv = nullptr, bool* qkv_done = nullptr) {
  const LayerW& L = e->layers[l];
  const int D = e->cfg.embed_dim, Hd = e->cfg.mlp_hidden, P = e->parts, S = e->split;
  const int M = B * N;
  if (xn_done != nullptr) *xn_done = false;
  if (qkv_done != nullptr) *qkv_done = false;
  if (!qkv_ready) {
    if (!xn_ready) TRY(run_layernorm(ws.X, L.ln1w, L.ln1b, ws.XN, 2LL * D, S, D, nullptr, 0, M, D, e->cfg.ln_eps, st, nullptr, e->f16));
    TRY(run_gemm(e, ws.XN, 2LL * D, L.wqkv.p, static_cast<long long>(D) * P, M, 3 * D, D, S, EPI_BIAS_BF16, L.bqkv, ws.QKV,
                 3LL * D * P, S, 3 * D, st, PC_GEMM_QKV));
  }
  TRY(run_attention(e, ws.QKV, 3LL * D * P, B, N, ws.CTX, static_cast<long long>(D) * P, st));
  // MLP of an act-split block (vitocm_set_layer_mode 1): norm2's output and the hidden activations are kept as (hi, lo) pairs and
  // fc1 / fc2 contract both halves against the single-precision weights (two MMAs per product) -- the rounding of these two
  // activations is where most of the CLS-row error of a 16-bit forward comes from (profiles/r02_precision_sim.txt)
  const bool mlp2 = !S && l < static_cast<int>(e->layer_mode.size()) && e->layer_mode[l] == 1;
  // proj + residual + norm2 + MLP + residual (+ the next block's norm1) in ONE kernel where an instantiation exists (single 16-bit
  // operands, D = 128 / 384): a row of the residual stream is read once and written once, norm2's output never reaches HBM
  if (!S && !mlp2) {
    // ... and the next block's QKV projection rides along (VITOCM_FUSE_QKV=0: the next norm1's rows go to HBM and its QKV GEMM runs)
    static const int fuse_qkv = [] { const char* v = getenv("VITOCM_FUSE_QKV"); return v ? atoi(v) : 1; }();
    const bool with_qkv = fuse_qkv && next_qkv != nullptr && next_ln_w != nullptr && qkv_done != nullptr;
    // LayerNorm affine parameters folded into W1 / Wqkv where vitocm_finalize_weights has prepared them (VITOCM_TAIL_FOLD=0: never)
    const bool fold = e->fold_valid;
    const int rct = run_block_tail(e, ws.CTX, static_cast<long long>(D) * P, L.wproj.p, static_cast<long long>(D) * P, L.bproj, L.ln2w, L.ln2b,
                                   fold ? L.w1_fold.p : L.w1.p, D, L.w2.p, Hd, M, D, Hd, fold ? L.b1_fold.as<float>() : L.b1, L.b2, ws.X,
                                   next_ln_w, next_ln_b, e->cfg.ln_eps, ws.XN, 2LL * D,
                                   with_qkv ? (fold ? next_qkv->wqkv_fold.p : next_qkv->wqkv.p) : nullptr, static_cast<long long>(D) * P,
                                   with_qkv ? (fold ? next_qkv->bqkv_fold.as<float>() : next_qkv->bqkv) : nullptr, ws.QKV, 3LL * D * P, st, false,
                                   nullptr, fold, fold);
    if (rct < 0) return rct;
    if (rct == 0) {
      if (with_qkv) *qkv_done = true;
      else if (xn_done != nullptr && next_ln_w != nullptr) *xn_done = true;
      return 0;
    }
  }
  // proj + residual (+ norm2 fused when possible)
  int rc = mlp2 ? 1 : run_gemm_ln(e, ws.CTX, static_cast<long long>(D) * P, L.wproj.p, static_cast<long long>(D) * P, M, D, D, L.bproj, ws.X,
                                  L.ln2w, L.ln2b, e->cfg.ln_eps, ws.XN, 2LL * D, st, PC_GEMM_PROJ);
  if (rc < 0) return rc;
  if (rc == 1) {
    TRY(run_gemm(e, ws.CTX, static_cast<long long>(D) * P, L.wproj.p, static_cast<long long>(D) * P, M, D, D, S,
                 EPI_BIAS_RESID_F32, L.bproj, ws.X, D, 0, 0, st, PC_GEMM_PROJ));
    TRY(run_layernorm(ws.X, L.ln2w, L.ln2b, ws.XN, 2LL * D, S || mlp2, D, nullptr, 0, M, D, e->cfg.ln_eps, st, nullptr, e->f16));
  }
  const int HP = mlp2 ? 2 : P;        // hidden activations: (hi | lo) in split engines and in act-split blocks
  const int mlp_in = S ? 1 : (mlp2 ? 2 : 0);
  // fc1 + GELU + fc2 + residual in one kernel where an instantiation exists (single 16-bit operands, D = 128 / 384): the hidden
  // activations never reach HBM
  if (!S && !mlp2) {
    rc = run_mlp_fused(e, ws.XN, 2LL * D, L.w1.p, D, L.w2.p, Hd, M, D, Hd, L.b1, L.b2, ws.X, st);
    if (rc < 0) return rc;
    if (rc == 0) return 0;
  }
  TRY(run_gemm(e, ws.XN, 2LL * D, L.w1.p, static_cast<long long>(D) * P, M, Hd, D, mlp_in, EPI_BIAS_GELU_BF16, L.b1, ws.HID,
               static_cast<long long>(Hd) * HP, S || mlp2, Hd, st, PC_GEMM_FC1));
  // fc2 + residual (+ the next block's norm1 fused when possible)
  rc = 1;
  if (next_ln_w != nullptr && !mlp2)
    rc = run_gemm_ln(e, ws.HID, static_cast<long long>(Hd) * P, L.w2.p, static_cast<long long>(Hd) * P, M, D, Hd, L.b2, ws.X, next_ln_w,
                     next_ln_b, e->cfg.ln_eps, ws.XN, 2LL * D, st, PC_GEMM_FC2);
  if (rc < 0) return rc;
  if (rc == 1) {
    TRY(run_gemm(e, ws.HID, static_cast<long long>(Hd) * HP, L.w2.p, static_cast<long long>(Hd) * P, M, D, Hd, mlp_in,
                 EPI_BIAS_RESID_F32, L.b2, ws.X, D, 0, 0, st, PC_GEMM_FC2));
  } else if (xn_done != nullptr) {
    *xn_done = true;
  }
  return 0;
}

int check_engine(const vitocm_engine* e) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  if (!e->finalized) return fail(VITOCM_ERR_STATE, "weights not finalized (call vitocm_finalize_weights)");
  return 0;
}

}  // namespace

// ====================================================================================== C ABI
extern "C" {

int vitocm_version(void) { return VITOCM_VERSION; }
const char* vitocm_last_error(void) { return g_err; }
int64_t vitocm_launch_count(void) { return g_launches.load(); }

int vitocm_profile_enable(int on) {
  g_prof_on = on != 0;
  return 0;
}
int vitocm_profile_classes(void) { return PC_COUNT; }
const char* vitocm_profile_class_name(int cls) { return (cls >= 0 && cls < PC_COUNT) ? kProfNames[cls] : ""; }
int vitocm_profile_read(double* ms, int64_t* counts, int nclasses) {
  if (ms == nullptr || counts == nullptr || nclasses < PC_COUNT) return fail(VITOCM_ERR_INVALID, "profile_read needs %d slots", PC_COUNT);
  for (int i = 0; i < nclasses; ++i) { ms[i] = 0.0; counts[i] = 0; }
  for (ProfRec& r : g_prof) {
    float t = 0.f;
    cudaEventSynchronize(r.b);
    cudaEventElapsedTime(&t, r.a, r.b);
    ms[r.cls] += t;
    counts[r.cls] += 1;
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  g_prof.clear();
  return 0;
}

int vitocm_create(const vitocm_config* cfg, vitocm_engine** out) {
  if (cfg == nullptr || out == nullptr) return fail(VITOCM_ERR_INVALID, "null argument");
  if (cfg->num_heads <= 0 || (cfg->embed_dim != cfg->num_heads * 64 && cfg->embed_dim != cfg->num_heads * 128))
    return fail(VITOCM_ERR_INVALID, "head_dim (embed_dim / num_heads) must be 64 or 128 (embed_dim %d, heads %d)", cfg->embed_dim, cfg->num_heads);
  if (cfg->mlp_hidden % 64 != 0 || cfg->depth < 1) return fail(VITOCM_ERR_INVALID, "bad mlp_hidden/depth");
  if (cfg->precision != VITOCM_BF16 && cfg->precision != VITOCM_FP32 && cfg->precision != VITOCM_FP16) return fail(VITOCM_ERR_INVALID, "bad precision");
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(VITOCM_ERR_CUDA, "libvitocm is built for sm_100a only (device is sm_%d%d)", prop.major, prop.minor);
  // One device per process (one process per GPU is the deployment model): the launch helpers cache per-function opt-ins
  // (cudaFuncSetAttribute, cluster occupancy) in process-wide statics, and those are per device.  A second device in the same
  // process is refused here instead of failing at its first launch.
  {
    static std::atomic<int> first_dev{-1};
    int expect = -1;
    if (!first_dev.compare_exchange_strong(expect, dev) && expect != dev)
      return fail(VITOCM_ERR_STATE, "libvitocm: engines of one process must live on one device (first engine on device %d, this one on %d)", expect, dev);
  }
  vitocm_engine* e = new vitocm_engine();
  e->cfg = *cfg;
  e->split = cfg->precision == VITOCM_FP32 ? 1 : 0;
  e->parts = e->split ? 2 : 1;
  e->f16 = cfg->precision == VITOCM_FP16 ? 1 : 0;
  e->num_sms = prop.multiProcessorCount;
  { const char* v = getenv("VITOCM_TAIL_FOLD"); e->tail_fold = v == nullptr ? 1 : atoi(v); }
  e->layers.resize(cfg->depth);
  e->layer_mode.assign(cfg->depth, 0);
  *out = e;
  return 0;
}

int vitocm_destroy(vitocm_engine* e) {
  delete e;
  return 0;
}

int vitocm_load_weight(vitocm_engine* e, const char* name, const float* host_data, int64_t numel) {
  if (e == nullptr || name == nullptr || host_data == nullptr || numel <= 0) return fail(VITOCM_ERR_INVALID, "bad argument");
  DevBuf* b = new DevBuf();
  int rc = b->alloc(static_cast<size_t>(numel) * 4);
  if (rc != 0) { delete b; return rc; }
  cudaError_t ce = cudaMemcpy(b->p, host_data, static_cast<size_t>(numel) * 4, cudaMemcpyHostToDevice);
  if (ce != cudaSuccess) { delete b; return fail(VITOCM_ERR_CUDA, "cudaMemcpy failed: %s", cudaGetErrorString(ce)); }
  auto it = e->master.find(name);
  if (it != e->master.end()) { delete it->second; it->second = b; } else { e->master[name] = b; }
  e->finalized = false;
  e->fold_valid = false;
  return 0;
}

static int repack_weights(vitocm_engine* e, cudaStream_t st) {
  const int D = e->cfg.embed_dim, Hd = e->cfg.mlp_hidden, P = e->parts, S = e->split;
  const int K = e->cfg.in_chans * e->cfg.patch_size * e->cfg.patch_size;
  auto need = [&](const std::string& n, long long cnt) -> int {
    if (e->numel(n) != cnt) return fail(VITOCM_ERR_STATE, "weight '%s' missing or wrong size (have %lld, need %lld)", n.c_str(), e->numel(n), cnt);
    return 0;
  };
  TRY(need("cls_token", D));
  TRY(need("patch_embed.proj.weight", static_cast<long long>(D) * K));
  TRY(need("patch_embed.proj.bias", D));
  TRY(need("norm.weight", D));
  TRY(need("norm.bias", D));
  auto pack = [&](DevBuf& dst, const float* src, int R, int C, int split) -> int {
    const int parts = split ? 2 : 1;
    TRY(dst.alloc(static_cast<size_t>(R) * C * parts * 2));
    split_weight_kernel<<<512, 256, 0, st>>>(src, dst.as<__nv_bfloat16>(), static_cast<long long>(C) * parts, split, C, R, C, e->f16);
    LAUNCH_CHECK();
    return 0;
  };
  std::vector<RepackEntry> entries;
  int total_tiles = 0;
  auto add_entry = [&](DevBuf& dst, DevBuf& dst_t, const float* src, int R, int C) -> int {
    TRY(dst.alloc(static_cast<size_t>(R) * C * 2));
    TRY(dst_t.alloc(static_cast<size_t>(R) * C * 2));
    RepackEntry en{src, dst.as<__nv_bfloat16>(), dst_t.as<__nv_bfloat16>(), R, C, total_tiles, (C + 31) / 32};
    total_tiles += ((R + 31) / 32) * en.tiles_c;
    entries.push_back(en);
    return 0;
  };
  if (e->cfg.in_chans > 1) {   // gray fast path (vitocm_forward_cls_attn_gray): filter folded over the channels
    const int pp = e->cfg.patch_size * e->cfg.patch_size;
    TRY(e->patch_w_gray_f32.alloc(static_cast<size_t>(D) * pp * 4));
    fold_patch_weight_kernel<<<(D * pp + 255) / 256, 256, 0, st>>>(e->w("patch_embed.proj.weight"), e->patch_w_gray_f32.as<float>(), D, e->cfg.in_chans, pp);
    LAUNCH_CHECK();
    TRY(pack(e->patch_w_gray, e->patch_w_gray_f32.as<float>(), D, pp, 1));
  }
  TRY(pack(e->patch_w, e->w("patch_embed.proj.weight"), D, K, 1));   // always hi | lo: K is tiny, keep the tokens fp32-grade
  for (int l = 0; l < e->cfg.depth; ++l) {
    const std::string pre = "blocks." + std::to_string(l) + ".";
    LayerW& L = e->layers[l];
    TRY(need(pre + "norm1.weight", D)); TRY(need(pre + "norm1.bias", D));
    TRY(need(pre + "norm2.weight", D)); TRY(need(pre + "norm2.bias", D));
    TRY(need(pre + "attn.qkv.weight", 3LL * D * D)); TRY(need(pre + "attn.qkv.bias", 3LL * D));
    TRY(need(pre + "attn.proj.weight", static_cast<long long>(D) * D)); TRY(need(pre + "attn.proj.bias", D));
    TRY(need(pre + "mlp.fc1.weight", static_cast<long long>(Hd) * D)); TRY(need(pre + "mlp.fc1.bias", Hd));
    TRY(need(pre + "mlp.fc2.weight", static_cast<long long>(D) * Hd)); TRY(need(pre + "mlp.fc2.bias", D));
    L.ln1w = e->w(pre + "norm1.weight"); L.ln1b = e->w(pre + "norm1.bias");
    L.ln2w = e->w(pre + "norm2.weight"); L.ln2b = e->w(pre + "norm2.bias");
    L.bqkv = e->w(pre + "attn.qkv.bias"); L.bproj = e->w(pre + "attn.proj.bias");
    L.b1 = e->w(pre + "mlp.fc1.bias"); L.b2 = e->w(pre + "mlp.fc2.bias");
    L.wqkv_f32 = e->w(pre + "attn.qkv.weight");
    if (S) {
      TRY(pack(L.wqkv, e->w(pre + "attn.qkv.weight"), 3 * D, D, S));
      TRY(pack(L.wproj, e->w(pre + "attn.proj.weight"), D, D, S));
      TRY(pack(L.w1, e->w(pre + "mlp.fc1.weight"), Hd, D, S));
      TRY(pack(L.w2, e->w(pre + "mlp.fc2.weight"), D, Hd, S));
    } else {   // bf16 engines: plain + transposed copies of all Linear weights in ONE launch (below)
      TRY(add_entry(L.wqkv, L.wqkv_t, e->w(pre + "attn.qkv.weight"), 3 * D, D));
      TRY(add_entry(L.wproj, L.wproj_t, e->w(pre + "attn.proj.weight"), D, D));
      TRY(add_entry(L.w1, L.w1_t, e->w(pre + "mlp.fc1.weight"), Hd, D));
      TRY(add_entry(L.w2, L.w2_t, e->w(pre + "mlp.fc2.weight"), D, Hd));
    }
    if (l == e->cfg.depth - 1) TRY(pack(L.wk_split, L.wqkv_f32 + static_cast<long long>(D) * D, D, D, 1));
  }
  (void)P;
  const long long dec_rows = static_cast<long long>(e->cfg.in_chans) * e->cfg.patch_size * e->cfg.patch_size;
  if (e->numel("decoder.0.weight") > 0) {   // MIM decoder (SSS/model.py:61-64), optional
    TRY(need("decoder.0.weight", dec_rows * D));
    TRY(need("decoder.0.bias", dec_rows));
    if (S) TRY(pack(e->dec_w, e->w("decoder.0.weight"), static_cast<int>(dec_rows), D, S));
    else TRY(add_entry(e->dec_w, e->dec_w_t, e->w("decoder.0.weight"), static_cast<int>(dec_rows), D));
  }
  if (e->patch_w_t_on && !S) {   // transposed copy only: the forward reads the filter as hi | lo (patch_w)
    TRY(e->patch_w_t.alloc(static_cast<size_t>(D) * K * 2));
    RepackEntry en{e->w("patch_embed.proj.weight"), nullptr, e->patch_w_t.as<__nv_bfloat16>(), D, K, total_tiles, (K + 31) / 32};
    total_tiles += ((D + 31) / 32) * en.tiles_c;
    entries.push_back(en);
  }
  if (!entries.empty()) {
    std::vector<const void*> key;
    for (const RepackEntry& en : entries) { key.push_back(en.src); key.push_back(en.dst); key.push_back(en.dst_t); }
    if (key != e->repack_key) {   // (re)upload the table only when a pointer changed; the steady-state refresh is one launch
      TRY(e->repack_table.alloc(entries.size() * sizeof(RepackEntry)));
      CUDA_TRY(cudaMemcpyAsync(e->repack_table.p, entries.data(), entries.size() * sizeof(RepackEntry), cudaMemcpyHostToDevice, st));
      CUDA_TRY(cudaStreamSynchronize(st));   // `entries` is a local
      e->repack_key = key;
      e->repack_entries = static_cast<int>(entries.size());
      e->repack_tiles = total_tiles;
    }
    repack_weights_kernel<<<e->repack_tiles, 256, 0, st>>>(e->repack_table.as<RepackEntry>(), e->repack_entries, e->f16);
    LAUNCH_CHECK();
  }
  return 0;
}

// LayerNorm affine parameters folded into the weights behind them, for the block-tail kernel of single 16-bit engines (LayerW::*_fold).
// Only vitocm_finalize_weights prepares them: a training engine refreshes its repacked weights every step and runs its forward through
// the separate kernels anyway.
static int fold_layernorm_weights(vitocm_engine* e, cudaStream_t st) {
  const int D = e->cfg.embed_dim, Hd = e->cfg.mlp_hidden;
  e->fold_valid = false;
  if (e->split || !e->tail_fold || (D != 128 && D != 384)) return 0;
  auto fold = [&](DevBuf& w_out, DevBuf& b_out, const float* w, const float* b, const float* g, const float* be, int R) -> int {
    TRY(w_out.alloc(static_cast<size_t>(R) * D * 2));
    TRY(b_out.alloc(static_cast<size_t>(R) * 4));
    fold_ln_weight_kernel<<<(R + 7) / 8, 256, 0, st>>>(w, b, g, be, w_out.as<__nv_bfloat16>(), b_out.as<float>(), R, D, e->f16);
    LAUNCH_CHECK();
    return 0;
  };
  for (int l = 0; l < e->cfg.depth; ++l) {
    const std::string pre = "blocks." + std::to_string(l) + ".";
    LayerW& L = e->layers[l];
    TRY(fold(L.w1_fold, L.b1_fold, e->w(pre + "mlp.fc1.weight"), L.b1, L.ln2w, L.ln2b, Hd));
    TRY(fold(L.wqkv_fold, L.bqkv_fold, L.wqkv_f32, L.bqkv, L.ln1w, L.ln1b, 3 * D));
  }
  e->fold_valid = true;
  return 0;
}

int vitocm_finalize_weights(vitocm_engine* e) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  TRY(repack_weights(e, nullptr));
  TRY(fold_layernorm_weights(e, nullptr));
  CUDA_TRY(cudaDeviceSynchronize());
  e->finalized = true;
  return 0;
}

int vitocm_refresh_weights(vitocm_engine* e, void* stream) {
  TRY(check_engine(e));
  e->fold_valid = false;   // the masters have changed: the block tail applies gamma / beta itself until the next vitocm_finalize_weights
  return repack_weights(e, static_cast<cudaStream_t>(stream));
}

int vitocm_bind_weight(vitocm_engine* e, const char* name, float* dev_data, int64_t numel) {
  if (e == nullptr || name == nullptr || dev_data == nullptr || numel <= 0) return fail(VITOCM_ERR_INVALID, "bad argument");
  if ((reinterpret_cast<uintptr_t>(dev_data) & 15) != 0) return fail(VITOCM_ERR_INVALID, "bound weight '%s' must be 16-byte aligned", name);
  auto it = e->master.find(name);
  DevBuf* b = it != e->master.end() ? it->second : (e->master[name] = new DevBuf());
  b->bind(dev_data, static_cast<size_t>(numel) * 4);
  e->finalized = false;
  e->fold_valid = false;
  return 0;
}

int vitocm_bind_grad(vitocm_engine* e, const char* name, float* dev_grad) {
  if (e == nullptr || name == nullptr) return fail(VITOCM_ERR_INVALID, "bad argument");
  if ((reinterpret_cast<uintptr_t>(dev_grad) & 15) != 0) return fail(VITOCM_ERR_INVALID, "bound gradient '%s' must be 16-byte aligned", name);
  if (dev_grad == nullptr) e->grads.erase(name); else e->grads[name] = dev_grad;
  return 0;
}


size_t vitocm_workspace_bytes(const vitocm_engine* e, int chunk_tiles, int n_tokens) {
  if (e == nullptr || chunk_tiles <= 0 || n_tokens <= 0) return 0;
  return carve(e, nullptr, chunk_tiles, n_tokens).total * e->lanes + 1024;
}

int vitocm_set_concurrency(vitocm_engine* e, int lanes) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  if (lanes < 1 || lanes > vitocm_engine::MAX_LANES) return fail(VITOCM_ERR_INVALID, "lanes must be in [1, %d]", vitocm_engine::MAX_LANES);
  if (e->ev_fork == nullptr) CUDA_TRY(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
  for (int i = 0; i < lanes - 1; ++i) {
    if (e->aux[i] == nullptr) CUDA_TRY(cudaStreamCreateWithFlags(&e->aux[i], cudaStreamNonBlocking));
    if (e->ev_join[i] == nullptr) CUDA_TRY(cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming));
  }
  e->lanes = lanes;
  return 0;
}

int vitocm_set_layer_mode(vitocm_engine* e, int layer, int mode) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  if (layer < 0 || layer >= e->cfg.depth) return fail(VITOCM_ERR_INVALID, "layer %d out of range", layer);
  if (mode != 0 && mode != 1) return fail(VITOCM_ERR_INVALID, "layer mode must be 0 (engine default) or 1 (MLP activations as hi/lo pairs)");
  if (mode == 1 && e->split) return fail(VITOCM_ERR_INVALID, "the fp32-parity engine already splits every operand");
  e->layer_mode[layer] = mode;
  return 0;
}

int vitocm_prepare_tokens(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask,
                          float* X, void* stream) {
  TRY(check_engine(e));
  return run_patch_embed(e, x, B, H, W, pos, mask, X, static_cast<cudaStream_t>(stream));
}

static int forward_rows(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const int* queries, int nq,
                        float* out_rows, float* k_out, void* ws, size_t ws_bytes, int chunk_tiles, void* stream, bool gray = false,
                        const MosaicSrc* mos = nullptr);

int vitocm_forward_cls_attn_gray(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, float* out_rows,
                                 void* ws, size_t ws_bytes, int chunk_tiles, void* stream) {
  return forward_rows(e, x, B, H, W, pos, nullptr, 1, out_rows, nullptr, ws, ws_bytes, chunk_tiles, stream, true);
}

// windows [t0, t0 + T) of an ny x nx grid
static int check_windows(const char* fn, int ny, int nx, int W, int S, int t0, int T) {
  if (ny < 1 || nx < 1 || S < 1 || W < 1 || t0 < 0 || T < 0 || static_cast<long long>(t0) + T > static_cast<long long>(ny) * nx)
    return fail(VITOCM_ERR_INVALID, "%s: bad window grid %dx%d W=%d S=%d tiles [%d, %lld)", fn, ny, nx, W, S, t0, static_cast<long long>(t0) + T);
  return 0;
}

int vitocm_forward_cls_attn_mosaic_grid(vitocm_engine* e, const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int ny, int nx, int W,
                                        int S, int t0, int T, const float* pos, float* out_rows, void* ws, size_t ws_bytes, int chunk_tiles,
                                        void* stream) {
  if (mosaic == nullptr) return fail(VITOCM_ERR_INVALID, "forward_cls_attn_mosaic: mosaic is NULL");
  TRY(check_windows("forward_cls_attn_mosaic", ny, nx, W, S, t0, T));
  const MosaicSrc src{mosaic, static_cast<long long>(pitch), mos_h, mos_w, nx, S, t0};
  return forward_rows(e, nullptr, T, W, W, pos, nullptr, 1, out_rows, nullptr, ws, ws_bytes, chunk_tiles, stream, true, &src);
}

int vitocm_forward_cls_attn_mosaic(vitocm_engine* e, const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int n, int W, int S, int t0,
                                   int T, const float* pos, float* out_rows, void* ws, size_t ws_bytes, int chunk_tiles, void* stream) {
  return vitocm_forward_cls_attn_mosaic_grid(e, mosaic, mos_h, mos_w, pitch, n, n, W, S, t0, T, pos, out_rows, ws, ws_bytes, chunk_tiles, stream);
}

int vitocm_forward_cls_attn(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, float* out_rows,
                            void* ws, size_t ws_bytes, int chunk_tiles, void* stream) {
  return forward_rows(e, x, B, H, W, pos, nullptr, 1, out_rows, nullptr, ws, ws_bytes, chunk_tiles, stream);
}

int vitocm_forward_query_attn(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const int* queries, int nq,
                              float* out_rows, float* k_out, void* ws, size_t ws_bytes, int chunk_tiles, void* stream) {
  if (queries == nullptr || nq < 1) return fail(VITOCM_ERR_INVALID, "forward_query_attn needs a device array of nq >= 1 token indices");
  return forward_rows(e, x, B, H, W, pos, queries, nq, out_rows, k_out, ws, ws_bytes, chunk_tiles, stream);
}

static int forward_rows(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const int* queries, int nq,
                        float* out_rows, float* k_out, void* ws, size_t ws_bytes, int chunk_tiles, void* stream, bool gray,
                        const MosaicSrc* mos) {
  TRY(check_engine(e));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int p = e->cfg.patch_size, D = e->cfg.embed_dim, heads = e->cfg.num_heads, C = gray ? 1 : e->cfg.in_chans;
  if (B <= 0) return 0;
  if (H % p || W % p) return fail(VITOCM_ERR_INVALID, "image %dx%d not a multiple of patch %d", H, W, p);
  const int N = (H / p) * (W / p) + 1;
  if (chunk_tiles <= 0) return fail(VITOCM_ERR_INVALID, "chunk_tiles must be positive");
  if (chunk_tiles > B) chunk_tiles = B;
  uint8_t* base = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<uintptr_t>(ws), 1024));
  const size_t avail = ws_avail(ws, base, ws_bytes);
  const size_t lane_bytes = carve(e, base, chunk_tiles, N).total;
  if (ws == nullptr || lane_bytes > avail) return fail(VITOCM_ERR_WORKSPACE, "workspace too small: need %zu, have %zu", lane_bytes + 1024, ws_bytes);
  // as many concurrent lanes as configured, as the workspace holds, and as there are chunks
  int lanes = e->lanes;
  if (static_cast<size_t>(lanes) * lane_bytes > avail) lanes = static_cast<int>(avail / lane_bytes);
  const int n_chunks = (B + chunk_tiles - 1) / chunk_tiles;
  if (lanes > n_chunks) lanes = n_chunks;
  const LayerW& last = e->layers[e->cfg.depth - 1];
  const int dh = D / heads;
  const size_t cls_smem = static_cast<size_t>(D + dh + N + 32) * sizeof(float);
  static size_t cls_smem_set[2] = {0, 0};
  if (cls_smem > 48 * 1024 && cls_smem > cls_smem_set[dh == 128]) {
    if (dh == 128) CUDA_TRY(cudaFuncSetAttribute(cls_attn_row_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(cls_smem)));
    else CUDA_TRY(cudaFuncSetAttribute(cls_attn_row_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(cls_smem)));
    cls_smem_set[dh == 128] = cls_smem;
  }
  cudaStream_t lane_st[vitocm_engine::MAX_LANES];
  Workspace lane_ws[vitocm_engine::MAX_LANES];
  for (int k = 0; k < lanes; ++k) {
    lane_st[k] = k == 0 ? st : e->aux[k - 1];
    lane_ws[k] = carve(e, base + static_cast<size_t>(k) * lane_bytes, chunk_tiles, N);
  }
  if (lanes > 1) {   // fork: the auxiliary streams start after everything already queued on the caller's stream
    CUDA_TRY(cudaEventRecord(e->ev_fork, st));
    for (int k = 1; k < lanes; ++k) CUDA_TRY(cudaStreamWaitEvent(lane_st[k], e->ev_fork, 0));
  }
  // groups of `lanes` chunks; launches are interleaved layer by layer so that the lanes advance together
  for (int g0 = 0; g0 < B; g0 += lanes * chunk_tiles) {
    int b0s[vitocm_engine::MAX_LANES], bcs[vitocm_engine::MAX_LANES], active = 0;
    for (int k = 0; k < lanes; ++k) {
      const int b0 = g0 + k * chunk_tiles;
      if (b0 >= B) break;
      b0s[k] = b0;
      bcs[k] = (B - b0 < chunk_tiles) ? (B - b0) : chunk_tiles;
      ++active;
    }
    for (int k = 0; k < active; ++k)
      if (mos != nullptr) {
        MosaicSrc part = *mos;
        part.t0 += b0s[k];
        TRY(run_patch_embed(e, nullptr, bcs[k], H, W, pos, nullptr, lane_ws[k].X, lane_st[k], true, &part));
      } else {
        TRY(run_patch_embed(e, x + static_cast<long long>(b0s[k]) * C * H * W, bcs[k], H, W, pos, nullptr, lane_ws[k].X, lane_st[k], gray));
      }
    bool xn_ready[vitocm_engine::MAX_LANES] = {false, false, false, false};
    bool qkv_ready[vitocm_engine::MAX_LANES] = {false, false, false, false};
    for (int l = 0; l + 1 < e->cfg.depth; ++l) {
      // the next block's norm1 rides on this block's fc2 epilogue -- except into the last block, whose K projection
      // wants the split-precision (hi | lo) normalised rows
      const bool chain = l + 2 < e->cfg.depth;
      for (int k = 0; k < active; ++k) {
        bool done = false, qdone = false;
        TRY(block_forward(e, l, lane_ws[k], bcs[k], N, lane_st[k], xn_ready[k], chain ? e->layers[l + 1].ln1w : nullptr,
                          chain ? e->layers[l + 1].ln1b : nullptr, &done, qkv_ready[k], chain ? &e->layers[l + 1] : nullptr, &qdone));
        xn_ready[k] = done;
        qkv_ready[k] = qdone;
      }
    }
    for (int k = 0; k < active; ++k) {
      // last block: LN1 (split) -> K projection in split precision -> fp32 K -> CLS-row softmax
      const Workspace& wsp = lane_ws[k];
      const int M = bcs[k] * N;
      float* KF = reinterpret_cast<float*>(wsp.HID);
      TRY(run_layernorm(wsp.X, last.ln1w, last.ln1b, wsp.XN, 2LL * D, 1, D, nullptr, 0, M, D, e->cfg.ln_eps, lane_st[k], nullptr, e->f16));
      TRY(run_gemm(e, wsp.XN, 2LL * D, last.wk_split.p, 2LL * D, M, D, D, 1, EPI_BIAS_F32, last.bqkv + D, KF, D, 0, 0, lane_st[k], PC_GEMM_KLAST));
      ProfScope prof(PC_CLSROW, lane_st[k]);
      dim3 grid(heads, bcs[k], nq);
      (dh == 128 ? cls_attn_row_kernel<128> : cls_attn_row_kernel<64>)<<<grid, 256, cls_smem, lane_st[k]>>>(
          wsp.X, last.ln1w, last.ln1b, e->cfg.ln_eps, last.wqkv_f32, last.bqkv, KF, out_rows + static_cast<long long>(b0s[k]) * heads * nq * N,
          N, D, heads, e->cfg.qk_scale, queries, nq);
      LAUNCH_CHECK();
      if (k_out != nullptr)   // last-block K features (SSS/analyse_attention.py:139-163, SSS/eval.py:186-202 cluster these)
        CUDA_TRY(cudaMemcpyAsync(k_out + static_cast<long long>(b0s[k]) * N * D, KF, static_cast<size_t>(M) * D * sizeof(float), cudaMemcpyDeviceToDevice,
                                 lane_st[k]));
    }
  }
  for (int k = 1; k < lanes; ++k) {   // join
    CUDA_TRY(cudaEventRecord(e->ev_join[k - 1], lane_st[k]));
    CUDA_TRY(cudaStreamWaitEvent(st, e->ev_join[k - 1], 0));
  }
  return 0;
}

int vitocm_block_forward(vitocm_engine* e, int layer, float* X, int B, int n_tokens, void* ws, size_t ws_bytes, void* stream) {
  TRY(check_engine(e));
  if (layer < 0 || layer >= e->cfg.depth) return fail(VITOCM_ERR_INVALID, "layer %d out of range", layer);
  void* base = reinterpret_cast<void*>(align_up(reinterpret_cast<uintptr_t>(ws), 1024));
  const size_t avail = ws_avail(ws, base, ws_bytes);
  Workspace wsp = carve(e, base, B, n_tokens);
  if (ws == nullptr || wsp.total > avail) return fail(VITOCM_ERR_WORKSPACE, "workspace too small: need %zu, have %zu", wsp.total + 1024, ws_bytes);
  wsp.X = X;  // operate in place on the caller's token stream
  return block_forward(e, layer, wsp, B, n_tokens, static_cast<cudaStream_t>(stream));
}

int vitocm_block_attn_probs(vitocm_engine* e, int layer, const float* X, int B, int n_tokens, float* attn, float* qkv_out,
                            void* ws, size_t ws_bytes, void* stream) {
  TRY(check_engine(e));
  if (layer < 0 || layer >= e->cfg.depth) return fail(VITOCM_ERR_INVALID, "layer %d out of range", layer);
  if (qkv_out == nullptr || attn == nullptr) return fail(VITOCM_ERR_INVALID, "attn and qkv_out are required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int D = e->cfg.embed_dim, P = e->parts, S = e->split, heads = e->cfg.num_heads, N = n_tokens;
  void* base = reinterpret_cast<void*>(align_up(reinterpret_cast<uintptr_t>(ws), 1024));
  const size_t avail = ws_avail(ws, base, ws_bytes);
  const Workspace wsp = carve(e, base, B, N);
  if (ws == nullptr || wsp.total > avail) return fail(VITOCM_ERR_WORKSPACE, "workspace too small: need %zu, have %zu", wsp.total + 1024, ws_bytes);
  const LayerW& L = e->layers[layer];
  const int M = B * N;
  TRY(run_layernorm(X, L.ln1w, L.ln1b, wsp.XN, 2LL * D, S, D, nullptr, 0, M, D, e->cfg.ln_eps, st, nullptr, e->f16));
  TRY(run_gemm(e, wsp.XN, 2LL * D, L.wqkv.p, static_cast<long long>(D) * P, M, 3 * D, D, S, EPI_BIAS_F32, L.bqkv, qkv_out, 3LL * D, 0, 0, st));
  const int dh = D / heads;
  const int kchunk = dh == 128 ? 128 : 256;
  int qrows = AP_QROWS;
  auto smem_for = [&](int qr) { return static_cast<size_t>(kchunk * (dh + 1) + qr * dh + static_cast<size_t>(qr) * N) * sizeof(float); };
  while (qrows > 1 && smem_for(qrows) > 200 * 1024) qrows >>= 1;
  const size_t smem = smem_for(qrows);
  if (smem > 220 * 1024) return fail(VITOCM_ERR_INVALID, "n_tokens=%d too large for attn_probs", N);
  static size_t smem_set[2] = {0, 0};
  if (smem > smem_set[dh == 128]) {
    if (dh == 128) CUDA_TRY(cudaFuncSetAttribute(attn_probs_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    else CUDA_TRY(cudaFuncSetAttribute(attn_probs_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    smem_set[dh == 128] = smem;
  }
  dim3 grid((N + qrows - 1) / qrows, heads, B);
  (dh == 128 ? attn_probs_kernel<128> : attn_probs_kernel<64>)<<<grid, 256, smem, st>>>(qkv_out, attn, N, D, heads, e->cfg.qk_scale, kchunk, qrows);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_mim_forward(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask, float* x_rec,
                       double* loss_sums, void* ws, size_t ws_bytes, int chunk_tiles, void* stream) {
  TRY(check_engine(e));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int p = e->cfg.patch_size, D = e->cfg.embed_dim, C = e->cfg.in_chans, P = e->parts, S = e->split;
  if (B <= 0) return 0;
  if (e->dec_w.p == nullptr) return fail(VITOCM_ERR_STATE, "MIM decoder weights (decoder.0.weight / decoder.0.bias) were never loaded");
  if (mask == nullptr || x_rec == nullptr || loss_sums == nullptr) return fail(VITOCM_ERR_INVALID, "mim_forward needs mask, x_rec and loss_sums");
  if (H % p || W % p) return fail(VITOCM_ERR_INVALID, "image %dx%d not a multiple of patch %d", H, W, p);
  const int n = (H / p) * (W / p), N = n + 1, ldy = C * p * p;
  if (ldy % 64 != 0) return fail(VITOCM_ERR_INVALID, "decoder width C*p*p=%d must be a multiple of 64", ldy);
  if (chunk_tiles <= 0) return fail(VITOCM_ERR_INVALID, "chunk_tiles must be positive");
  if (chunk_tiles > B) chunk_tiles = B;
  void* base = reinterpret_cast<void*>(align_up(reinterpret_cast<uintptr_t>(ws), 1024));
  const size_t avail = ws_avail(ws, base, ws_bytes);
  const Workspace wsp = carve(e, base, chunk_tiles, N);
  if (ws == nullptr || wsp.total > avail) return fail(VITOCM_ERR_WORKSPACE, "workspace too small: need %zu, have %zu", wsp.total + 1024, ws_bytes);
  CUDA_TRY(cudaMemsetAsync(loss_sums, 0, 2 * sizeof(double), st));
  // decoder output Y [M][C p^2] fp32 lives where QKV / CTX / HID are (all idle after the last block); it must end inside the carve-up
  float* Y = reinterpret_cast<float*>(wsp.QKV);
  if (static_cast<size_t>(chunk_tiles) * N * ldy * sizeof(float) > wsp.total - (reinterpret_cast<uintptr_t>(wsp.QKV) - reinterpret_cast<uintptr_t>(base)))
    return fail(VITOCM_ERR_WORKSPACE, "decoder output of width %d does not fit behind the token stream of this workspace", ldy);
  for (int b0 = 0; b0 < B; b0 += chunk_tiles) {
    const int bc = (B - b0 < chunk_tiles) ? (B - b0) : chunk_tiles;
    const int M = bc * N;
    const float* xc = x + static_cast<long long>(b0) * C * H * W;
    const float* mc = mask + static_cast<long long>(b0) * n;
    // VisionTransformerForSimMIM.forward (SSS/model.py:25-53): patch embed + mask-token mix + cls + pos, all blocks, norm
    TRY(run_patch_embed(e, xc, bc, H, W, pos, mc, wsp.X, st));
    for (int l = 0; l < e->cfg.depth; ++l) TRY(block_forward(e, l, wsp, bc, N, st));
    TRY(run_layernorm(wsp.X, e->w("norm.weight"), e->w("norm.bias"), wsp.XN, 2LL * D, S, D, nullptr, 0, M, D, e->cfg.ln_eps, st, nullptr, e->f16));
    // decoder: 1x1 conv D -> C p^2 == per-token linear (model.py:61-64); CLS rows are computed and ignored
    TRY(run_gemm(e, wsp.XN, 2LL * D, e->dec_w.p, static_cast<long long>(D) * P, M, ldy, D, S, EPI_BIAS_F32, e->w("decoder.0.bias"), Y,
                 ldy, 0, 0, st));
    const long long total = static_cast<long long>(bc) * C * H * W;
    long long grid = (total + 255) / 256;
    if (grid > 148LL * 16) grid = 148LL * 16;
    mim_shuffle_loss_kernel<<<static_cast<int>(grid), 256, 0, st>>>(Y, xc, mc, x_rec + static_cast<long long>(b0) * C * H * W, loss_sums, bc, C, H,
                                                                     W, p);
    LAUNCH_CHECK();
  }
  return 0;
}

int vitocm_final_norm(vitocm_engine* e, const float* X, float* out, int M, void* stream) {
  TRY(check_engine(e));
  const int D = e->cfg.embed_dim;
  return run_layernorm(X, e->w("norm.weight"), e->w("norm.bias"), nullptr, 0, 0, 0, out, D, M, D, e->cfg.ln_eps,
                       static_cast<cudaStream_t>(stream));
}

// ------------------------------------------------------------------------------ post-processing
int vitocm_head_mean(const float* rows, float* lowres, int T, int heads, int n_tokens, int mode, void* stream) {
  if (T <= 0) return 0;
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  head_mean_kernel<<<T, 256, 0, static_cast<cudaStream_t>(stream)>>>(rows, lowres, heads, n_tokens, mode);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_attn_cummass(const float* rows, int T, int heads, int n_tokens, float threshold, uint8_t* mask, float* up, int lh, int lw,
                        int patch, void* stream) {
  if (T <= 0) return 0;
  if (rows == nullptr || mask == nullptr || heads < 1 || n_tokens < 2) return fail(VITOCM_ERR_INVALID, "attn_cummass: bad argument");
  if (up != nullptr && (lh * lw != n_tokens - 1 || patch < 1)) return fail(VITOCM_ERR_INVALID, "attn_cummass: lh * lw must equal n_tokens - 1 for the upsampled output");
  int npow2 = 32;
  while (npow2 < n_tokens - 1) npow2 <<= 1;
  if (npow2 > CM_MAX) return fail(VITOCM_ERR_INVALID, "attn_cummass: at most %d patches per tile", CM_MAX);
  const size_t smem = static_cast<size_t>(2 * npow2 + 8) * sizeof(float);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProfScope prof(PC_POST, st);
  // `cumval > (1 - threshold)`: the Python double 1 - th is compared in the tensor's dtype, fp32
  const float keep_above = static_cast<float>(1.0 - static_cast<double>(threshold));
  cummass_kernel<<<T * heads, 256, smem, st>>>(rows, heads, n_tokens, npow2, keep_above, mask, up, lh, lw, patch);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_tile_threshold(const float* lowres, const float* x, int T, int C, int S, int lh, int lw, uint8_t* masks,
                          int* thresholds, float* att_out, const float* att_in, const uint8_t* img_in, void* stream) {
  if (T <= 0) return 0;
  if (lowres == nullptr && att_in == nullptr) return fail(VITOCM_ERR_INVALID, "tile_threshold needs lowres or att_in");
  if (x == nullptr && img_in == nullptr) return fail(VITOCM_ERR_INVALID, "tile_threshold needs x or img_in");
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  tile_threshold_kernel<<<T, 512, 0, static_cast<cudaStream_t>(stream)>>>(lowres, x, C, S, lh, lw, masks, thresholds, att_out, att_in, img_in, nullptr);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_tile_threshold_aux(const float* lowres, const float* x, int T, int C, int S, int lh, int lw, uint8_t* masks,
                              int* thresholds, float* att_out, const float* att_in, const uint8_t* img_in, uint8_t* aux, void* stream) {
  if (T <= 0) return 0;
  if (lowres == nullptr && att_in == nullptr) return fail(VITOCM_ERR_INVALID, "tile_threshold needs lowres or att_in");
  if (x == nullptr && img_in == nullptr) return fail(VITOCM_ERR_INVALID, "tile_threshold needs x or img_in");
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  tile_threshold_kernel<<<T, 512, 0, static_cast<cudaStream_t>(stream)>>>(lowres, x, C, S, lh, lw, masks, thresholds, att_out, att_in, img_in, aux);
  LAUNCH_CHECK();
  return 0;
}

static int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  const long long cap = 148LL * 16;
  return static_cast<int>(g < 1 ? 1 : (g > cap ? cap : g));
}

int vitocm_extract_tiles_grid(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int ny, int nx, int W, int S, int t0, int T, int C,
                              float* x, void* stream) {
  if (T <= 0) return 0;
  TRY(check_windows("extract_tiles", ny, nx, W, S, t0, T));
  const long long total = static_cast<long long>(T) * W * W;
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  extract_tiles_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(mosaic, mos_h, mos_w, pitch, nx, W, S, t0, T, C, x);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_extract_tiles(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int n, int W, int S, int t0, int T, int C,
                         float* x, void* stream) {
  return vitocm_extract_tiles_grid(mosaic, mos_h, mos_w, pitch, n, n, W, S, t0, T, C, x, stream);
}

// Row-organised mosaic kernels: grid.x covers one row in groups of 256 * V pixels (V = 4 when every row of every buffer is
// 16-byte aligned, i.e. Ex % 4 == 0 and aligned bases, else 1); grid.y strides over the rows of the band, ~8 blocks per SM
struct StitchLaunch { dim3 grid; int V; };
static StitchLaunch stitch_launch(int E /*row length Ex*/, int rows, int num_sms, std::initializer_list<const void*> f32_ptrs, std::initializer_list<const void*> u8_ptrs) {
  bool vec = (E % 4) == 0;
  for (const void* p : f32_ptrs) if (p != nullptr && (reinterpret_cast<uintptr_t>(p) & 15) != 0) vec = false;
  for (const void* p : u8_ptrs) if (p != nullptr && (reinterpret_cast<uintptr_t>(p) & 3) != 0) vec = false;
  StitchLaunch L;
  L.V = vec ? 4 : 1;
  const int gx = (E + 256 * L.V - 1) / (256 * L.V);
  int gy = (num_sms * 8 + gx - 1) / gx;
  if (gy > rows) gy = rows;
  if (gy < 1) gy = 1;
  L.grid = dim3(gx, gy);
  return L;
}
static int device_sms() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  return sms;
}

// kernels that evaluate the stitched map from the low-res maps keep a W-entry coefficient table in shared memory
static int check_tab(const void* map_in, int W) {
  if (map_in == nullptr && W > ST_MAX_W) return fail(VITOCM_ERR_INVALID, "window %d exceeds the stitch kernels' limit of %d pixels", W, ST_MAX_W);
  return 0;
}

static StitchGeom make_geom(int ny, int nx, int W, int S, int lh, int lw) {
  StitchGeom g;
  g.ny = ny; g.nx = nx; g.W = W; g.S = S; g.step = W - S; g.Ey = (ny - 1) * S + W; g.Ex = (nx - 1) * S + W; g.lh = lh; g.lw = lw;
  g.scale = static_cast<double>(lw) / static_cast<double>(W);
  return g;
}
static int check_geom(int ny, int nx, int W, int S, int y_begin, int y_end) {
  if (ny < 1 || nx < 1 || S < 1 || W <= S) return fail(VITOCM_ERR_INVALID, "bad sliding-window geometry %dx%d W=%d S=%d", ny, nx, W, S);
  if (W > 4 * S) return fail(VITOCM_ERR_INVALID, "sliding-window geometry W=%d S=%d: at most four windows may overlap (W <= 4 S)", W, S);
  const long long Ey = static_cast<long long>(ny - 1) * S + W, Ex = static_cast<long long>(nx - 1) * S + W;
  if (Ey > INT_MAX || Ex > INT_MAX || Ey * Ex > (1LL << 40))
    return fail(VITOCM_ERR_INVALID, "sliding-window grid %dx%d at stride %d: extent %lldx%lld too large", ny, nx, S, Ey, Ex);
  if (y_begin < 0 || y_end > Ey || y_begin > y_end) return fail(VITOCM_ERR_INVALID, "bad row band [%d,%d) for extent %lld", y_begin, y_end, Ey);
  return 0;
}

int vitocm_stitch_gray_grid(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int ny, int nx, int W, int S, const double* wtab,
                            int y_begin, int y_end, uint8_t* out, void* stream) {
  TRY(check_geom(ny, nx, W, S, y_begin, y_end));
  if (y_end == y_begin) return 0;
  const StitchGeom g = make_geom(ny, nx, W, S, 1, 1);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProfScope prof(PC_POST, st);
  const StitchLaunch L = stitch_launch(g.Ex, y_end - y_begin, device_sms(), {}, {out});
  static const int strip = [] { const char* v = getenv("VITOCM_STITCH_STRIP"); return v == nullptr ? 1 : atoi(v); }();
  if (strip) {   // column-strip kernels (VITOCM_STITCH_STRIP=0: the row-organised ones)
    const dim3 grid((g.Ex + SG_THREADS * L.V - 1) / (SG_THREADS * L.V), (y_end - y_begin + SG_ROWS - 1) / SG_ROWS);
    if (L.V == 4 && W <= 2 * S) stitch_gray_strip_kernel<4, 2><<<grid, SG_THREADS, 0, st>>>(mosaic, mos_h, mos_w, pitch, g, wtab, y_begin, y_end, out);
    else if (L.V == 4) stitch_gray_strip_kernel<4, 4><<<grid, SG_THREADS, 0, st>>>(mosaic, mos_h, mos_w, pitch, g, wtab, y_begin, y_end, out);
    else if (W <= 2 * S) stitch_gray_strip_kernel<1, 2><<<grid, SG_THREADS, 0, st>>>(mosaic, mos_h, mos_w, pitch, g, wtab, y_begin, y_end, out);
    else stitch_gray_strip_kernel<1, 4><<<grid, SG_THREADS, 0, st>>>(mosaic, mos_h, mos_w, pitch, g, wtab, y_begin, y_end, out);
    LAUNCH_CHECK();
    return 0;
  }
  if (L.V == 4) stitch_gray_kernel<4><<<L.grid, 256, 0, st>>>(mosaic, mos_h, mos_w, pitch, g, wtab, y_begin, y_end, out);
  else stitch_gray_kernel<1><<<L.grid, 256, 0, st>>>(mosaic, mos_h, mos_w, pitch, g, wtab, y_begin, y_end, out);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_stitch_gray(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int n, int W, int S, const double* wtab,
                       int y_begin, int y_end, uint8_t* out, void* stream) {
  return vitocm_stitch_gray_grid(mosaic, mos_h, mos_w, pitch, n, n, W, S, wtab, y_begin, y_end, out, stream);
}

int vitocm_minmax_init(int* minmax_ord, void* stream) {
  const int init[2] = {0x7fffffff, static_cast<int>(0x80000000u)};
  CUDA_TRY(cudaMemcpyAsync(minmax_ord, init, sizeof(init), cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
  return 0;
}

int vitocm_stitch_minmax_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab, int y_begin, int y_end,
                              int* minmax_ord, float* map_out, const float* map_in, void* stream) {
  TRY(check_geom(ny, nx, W, S, y_begin, y_end));
  TRY(check_tab(map_in, W));
  if (y_end == y_begin) return 0;
  const StitchGeom g = make_geom(ny, nx, W, S, lh, lw);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProfScope prof(PC_POST, st);
  // stitched from the low-res maps: column-strip kernel (VITOCM_STITCH_STRIP=0: the row-organised one)
  static const int strip = [] { const char* v = getenv("VITOCM_STITCH_STRIP"); return v == nullptr ? 1 : atoi(v); }();
  if (map_in == nullptr && strip) {
    const dim3 grid((g.Ex + SC_THREADS - 1) / SC_THREADS, (y_end - y_begin + SC_ROWS - 1) / SC_ROWS);
    if (W <= 2 * S) stitch_strip_kernel<2><<<grid, SC_THREADS, 0, st>>>(lowres, g, wtab, y_begin, y_end, minmax_ord, map_out);
    else stitch_strip_kernel<4><<<grid, SC_THREADS, 0, st>>>(lowres, g, wtab, y_begin, y_end, minmax_ord, map_out);
    LAUNCH_CHECK();
    return 0;
  }
  const StitchLaunch L = stitch_launch(g.Ex, y_end - y_begin, device_sms(), {map_out, map_in}, {});
  if (L.V == 4) stitch_minmax_kernel<4><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, y_begin, y_end, minmax_ord, map_out, map_in);
  else stitch_minmax_kernel<1><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, y_begin, y_end, minmax_ord, map_out, map_in);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_stitch_minmax(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab, int y_begin, int y_end,
                         int* minmax_ord, float* map_out, const float* map_in, void* stream) {
  return vitocm_stitch_minmax_grid(lowres, n, n, W, S, lh, lw, wtab, y_begin, y_end, minmax_ord, map_out, map_in, stream);
}

int vitocm_stitch_hist_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                            const int* minmax_ord, int y_begin, int y_end, uint64_t* hists, const float* map_in, void* stream) {
  TRY(check_geom(ny, nx, W, S, y_begin, y_end));
  TRY(check_tab(map_in, W));
  if (y_end == y_begin) return 0;
  const StitchGeom g = make_geom(ny, nx, W, S, lh, lw);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProfScope prof(PC_POST, st);
  const StitchLaunch L = stitch_launch(g.Ex, y_end - y_begin, device_sms(), {map_in}, {gray});
  unsigned long long* h = reinterpret_cast<unsigned long long*>(hists);
  if (L.V == 4) stitch_hist_kernel<4><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, gray, minmax_ord, y_begin, y_end, h, map_in);
  else stitch_hist_kernel<1><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, gray, minmax_ord, y_begin, y_end, h, map_in);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_stitch_hist(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                       const int* minmax_ord, int y_begin, int y_end, uint64_t* hists, const float* map_in, void* stream) {
  return vitocm_stitch_hist_grid(lowres, n, n, W, S, lh, lw, wtab, gray, minmax_ord, y_begin, y_end, hists, map_in, stream);
}

int vitocm_otsu(const uint64_t* hists, int nhist, int* thresholds, void* stream) {
  if (nhist <= 0) return 0;
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  otsu_block_kernel<<<nhist, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const unsigned long long*>(hists), thresholds);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_stitch_mask_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                            const int* minmax_ord, const int* thr, int y_begin, int y_end, uint8_t* th, uint8_t* th2, uint8_t* th3,
                            const float* map_in, void* stream) {
  TRY(check_geom(ny, nx, W, S, y_begin, y_end));
  TRY(check_tab(map_in, W));
  if (y_end == y_begin) return 0;
  const StitchGeom g = make_geom(ny, nx, W, S, lh, lw);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProfScope prof(PC_POST, st);
  const StitchLaunch L = stitch_launch(g.Ex, y_end - y_begin, device_sms(), {map_in}, {gray, th, th2, th3});
  if (L.V == 4) stitch_mask_kernel<4><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, gray, minmax_ord, thr, y_begin, y_end, th, th2, th3, map_in);
  else stitch_mask_kernel<1><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, gray, minmax_ord, thr, y_begin, y_end, th, th2, th3, map_in);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_stitch_mask(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                       const int* minmax_ord, const int* thr, int y_begin, int y_end, uint8_t* th, uint8_t* th2, uint8_t* th3,
                       const float* map_in, void* stream) {
  return vitocm_stitch_mask_grid(lowres, n, n, W, S, lh, lw, wtab, gray, minmax_ord, thr, y_begin, y_end, th, th2, th3, map_in, stream);
}

int vitocm_stitch_result_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                              const int* minmax_ord, int y_begin, int y_end, uint8_t* result, uint8_t* att_u8, const float* map_in,
                              void* stream) {
  TRY(check_geom(ny, nx, W, S, y_begin, y_end));
  TRY(check_tab(map_in, W));
  if (y_end == y_begin) return 0;
  const StitchGeom g = make_geom(ny, nx, W, S, lh, lw);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ProfScope prof(PC_POST, st);
  const StitchLaunch L = stitch_launch(g.Ex, y_end - y_begin, device_sms(), {map_in}, {gray});
  if (L.V == 4) stitch_result_kernel<4><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, gray, minmax_ord, y_begin, y_end, result, att_u8, map_in);
  else stitch_result_kernel<1><<<L.grid, ST_THREADS, 0, st>>>(lowres, g, wtab, gray, minmax_ord, y_begin, y_end, result, att_u8, map_in);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_stitch_result(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                         const int* minmax_ord, int y_begin, int y_end, uint8_t* result, uint8_t* att_u8, const float* map_in, void* stream) {
  return vitocm_stitch_result_grid(lowres, n, n, W, S, lh, lw, wtab, gray, minmax_ord, y_begin, y_end, result, att_u8, map_in, stream);
}

int vitocm_concat_crops_grid_f32(const float* crops, int ny, int nx, int W, int S, const double* wtab, float* out, void* stream) {
  TRY(check_geom(ny, nx, W, S, 0, 0));
  const StitchGeom g = make_geom(ny, nx, W, S, 1, 1);
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  concat_crops_f32_kernel<<<grid_for(static_cast<long long>(g.Ey) * g.Ex, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(crops, g, wtab, out);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_concat_crops_f32(const float* crops, int n, int W, int S, const double* wtab, float* out, void* stream) {
  return vitocm_concat_crops_grid_f32(crops, n, n, W, S, wtab, out, stream);
}

int vitocm_concat_crops_grid_u8(const uint8_t* crops, int ny, int nx, int W, int S, int C, const double* wtab, uint8_t* out, void* stream) {
  TRY(check_geom(ny, nx, W, S, 0, 0));
  const StitchGeom g = make_geom(ny, nx, W, S, 1, 1);
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  concat_crops_u8_kernel<<<grid_for(static_cast<long long>(g.Ey) * g.Ex * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(crops, g, C, wtab, out);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_concat_crops_u8(const uint8_t* crops, int n, int W, int S, int C, const double* wtab, uint8_t* out, void* stream) {
  return vitocm_concat_crops_grid_u8(crops, n, n, W, S, C, wtab, out, stream);
}

int vitocm_crop_u8(const uint8_t* img, int img_h, int img_w, int C, int ny, int nx, int W, int S, uint8_t* crops, void* stream) {
  if (ny <= 0 || nx <= 0) return 0;
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  crop_u8_kernel<<<grid_for(static_cast<long long>(ny) * nx * W * W * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(img, img_h, img_w, C, ny, nx, W, S, crops);
  LAUNCH_CHECK();
  return 0;
}

static int overlap_geom(int n, int W, int stride, OverlapGeom* g) {
  const long long V = 2LL * stride;
  if (n < 1 || stride < 1 || V >= W) return fail(VITOCM_ERR_INVALID, "bad overlap geometry n=%d W=%d stride=%d (needs 0 < 2*stride < W)", n, W, stride);
  g->n = n; g->W = W; g->V = static_cast<int>(V); g->step = W - g->V; g->E = W + (n - 1) * g->step;
  return 0;
}

int vitocm_concat_crops_overlap_f32(const float* crops, int n, int W, int stride, float* out, void* stream) {
  OverlapGeom g;
  TRY(overlap_geom(n, W, stride, &g));
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  concat_crops_overlap_kernel<float><<<grid_for(static_cast<long long>(g.E) * g.E, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(crops, g, 1, out);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_concat_crops_overlap_u8(const uint8_t* crops, int n, int W, int stride, int C, uint8_t* out, void* stream) {
  OverlapGeom g;
  TRY(overlap_geom(n, W, stride, &g));
  if (C < 1) return fail(VITOCM_ERR_INVALID, "bad channel count %d", C);
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  concat_crops_overlap_kernel<uint8_t><<<grid_for(static_cast<long long>(g.E) * g.E * C, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(crops, g, C, out);
  LAUNCH_CHECK();
  return 0;
}

int vitocm_concat_grid_f32(const float* src, int B, int cr, int C, int c0, int h, int w, float* dst, void* stream) {
  if (B < 0 || cr < 1 || C < 1 || c0 < 0 || c0 >= C || h < 1 || w < 1) return fail(VITOCM_ERR_INVALID, "bad crop grid B=%d cr=%d C=%d c0=%d h=%d w=%d", B, cr, C, c0, h, w);
  if (B == 0) return 0;
  ProfScope prof(PC_POST, static_cast<cudaStream_t>(stream));
  concat_grid_f32_kernel<<<grid_for(static_cast<long long>(B) * cr * h * cr * w, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, B, cr, C, c0, h, w, dst);
  LAUNCH_CHECK();
  return 0;
}

// ------------------------------------------------------------------------------ kernel-level entry points
int vitocm_gemm(vitocm_engine* e, const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K, int split_in,
                int epilogue, const float* bias, void* out, int64_t ldo, int split_out, int lo_off, void* stream) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  return run_gemm(e, A, lda, B, ldb, M, N, K, split_in, epilogue, bias, out, ldo, split_out, lo_off, static_cast<cudaStream_t>(stream));
}

int vitocm_gemm_ln(vitocm_engine* e, const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K, const float* bias,
                   float* X, const float* gamma, const float* beta, void* XN, int64_t ld_xn, void* stream) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  const int rc = run_gemm_ln(e, A, lda, B, ldb, M, N, K, bias, X, gamma, beta, e->cfg.ln_eps, XN, ld_xn, static_cast<cudaStream_t>(stream), PC_OTHER);
  if (rc == 1) return fail(VITOCM_ERR_INVALID, "no fused GEMM+LayerNorm instantiation for N=%d (needs N/128 in {1,2,3,4,6}, bf16 engine)", N);
  return rc;
}

int vitocm_mlp_fused(vitocm_engine* e, const void* XN, int64_t ld_xn, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2, int M, int D,
                     int hidden, const float* bias1, const float* bias2, float* X, void* stream) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  const int rc = run_mlp_fused(e, XN, ld_xn, W1, ldw1, W2, ldw2, M, D, hidden, bias1, bias2, X, reinterpret_cast<cudaStream_t>(stream), true);
  if (rc == 1) return fail(VITOCM_ERR_INVALID, "fused MLP: no instantiation for D=%d hidden=%d in this engine mode", D, hidden);
  return rc;
}
int vitocm_mlp_fused_timeline(vitocm_engine* e, const void* XN, int64_t ld_xn, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2,
                              int M, int D, int hidden, const float* bias1, const float* bias2, float* X, int64_t* stamps, void* stream) {
  if (e == nullptr || stamps == nullptr) return fail(VITOCM_ERR_INVALID, "null engine / stamps");
  const int rc = run_mlp_fused(e, XN, ld_xn, W1, ldw1, W2, ldw2, M, D, hidden, bias1, bias2, X, reinterpret_cast<cudaStream_t>(stream), true,
                               reinterpret_cast<long long*>(stamps));
  if (rc == 1) return fail(VITOCM_ERR_INVALID, "fused MLP: no instantiation for D=%d hidden=%d in this engine mode", D, hidden);
  return rc;
}
int vitocm_block_tail(vitocm_engine* e, const void* CTX, int64_t ld_ctx, const void* Wp, int64_t ldwp, const float* bias_p, const float* ln2_w,
                      const float* ln2_b, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2, int M, int D, int hidden, const float* bias1,
                      const float* bias2, float* X, const float* next_ln_w, const float* next_ln_b, void* XN, int64_t ld_xn, const void* Wqkv,
                      int64_t ldwqkv, const float* bias_qkv, void* QKV, int64_t ld_qkv, int64_t* stamps, void* stream) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  // diagnostics (tools/tail_timeline.py): VITOCM_TAIL_ASSUME_FOLDED=1 runs the kernel as the engine's forward does after
  // vitocm_finalize_weights -- the caller's W1 / bias1 / Wqkv / bias_qkv are taken to carry the LayerNorm affine parameters already
  static const bool folded = [] { const char* v = getenv("VITOCM_TAIL_ASSUME_FOLDED"); return v != nullptr && atoi(v) != 0; }();
  const int rc = run_block_tail(e, CTX, ld_ctx, Wp, ldwp, bias_p, ln2_w, ln2_b, W1, ldw1, W2, ldw2, M, D, hidden, bias1, bias2, X, next_ln_w,
                                next_ln_b, e->cfg.ln_eps, XN, ld_xn, Wqkv, ldwqkv, bias_qkv, QKV, ld_qkv, reinterpret_cast<cudaStream_t>(stream), true,
                                reinterpret_cast<long long*>(stamps), folded, folded);
  if (rc == 1) return fail(VITOCM_ERR_INVALID, "block tail: no instantiation for D = %d, hidden = %d on this engine (or inconsistent optional arguments)", D, hidden);
  return rc;
}
int vitocm_attention(vitocm_engine* e, const void* qkv, int64_t ld, int B, int n_tokens, void* ctx, int64_t ldo, void* stream) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  return run_attention(e, qkv, ld, B, n_tokens, ctx, ldo, static_cast<cudaStream_t>(stream));
}

int vitocm_attention_timeline(vitocm_engine* e, const void* qkv, int64_t ld, int B, int n_tokens, void* ctx, int64_t ldo,
                              int64_t* stamps, void* stream) {
  if (e == nullptr || stamps == nullptr) return fail(VITOCM_ERR_INVALID, "null argument");
  return run_attention(e, qkv, ld, B, n_tokens, ctx, ldo, static_cast<cudaStream_t>(stream), reinterpret_cast<long long*>(stamps));
}

int vitocm_layernorm(vitocm_engine* e, const float* X, const float* gamma, const float* beta, void* out_bf16, int64_t ldo,
                     int split, int lo_off, int M, void* stream) {
  if (e == nullptr) return fail(VITOCM_ERR_INVALID, "null engine");
  return run_layernorm(X, gamma, beta, out_bf16, ldo, split, lo_off, nullptr, 0, M, e->cfg.embed_dim, e->cfg.ln_eps,
                       static_cast<cudaStream_t>(stream), nullptr, e->f16);
}

}  // extern "C"

#include "train_api.inc"
