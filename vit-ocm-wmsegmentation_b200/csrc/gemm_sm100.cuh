// Persistent, warp-specialised tcgen05 GEMM for sm_100a:
//     C[M,N] = epilogue( sum_t A[:, a_koff[t] : +K] * B[:, b_koff[t] : +K]^T )
// A [M, lda] and B [N, ldb] are bf16, K-major (row-major with K contiguous), staged by TMA into
// 128B-swizzled shared-memory tiles; accumulators live in TMEM (2 stages, so the epilogue of
// tile i overlaps the main loop of tile i+1).  `nterms` = 3 with hi/lo operand halves gives the
// split-bf16 ("fp32 mode") product  hi*hi + hi*lo + lo*hi  in the same kernel.
//
// Replaces, on the reference path, nn.Linear at SSS/dino/vision_transformer.py:58,61 (fc1/fc2),
// :80 (qkv), :88 (proj) with their bias / GELU (:59) / residual (:110-111) fused as epilogues, and
// (A_PATCH) the patch-embedding Conv2d at :127-131 + prepare_tokens :203-207 as an im2col-free GEMM:
// the producer warps read NCHW fp32 pixels and write the bf16 K-major A tile straight into the
// swizzled smem layout the MMA reads; nothing is materialised in HBM.
//
// Epilogue: TMEM -> registers (lane = row) -> bias / GELU -> per-warp swizzled smem box -> one TMA
// store per 32x32 chunk (cp.async.bulk.tensor, rows beyond M clipped by the tensor map).  The fp32
// residual epilogue uses the TMA reduce-add (cp.reduce.async.bulk.tensor .add): x += acc + bias is
// performed by the L2, so the residual stream is never read back into the SM.
//
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, warps 4..11(15) = epilogue
// (A_PATCH: warps 2, 3 and six more warps after the epilogue warps are the A producers) (lane quadrant = warp % 4,
// column group = (warp - 4) / 4).
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace vitocm {

enum GemmEpilogue : int {
  EPI_BIAS_BF16 = 0,       // out_bf16 = acc + bias                (qkv / k projection)
  EPI_BIAS_GELU_BF16 = 1,  // out_bf16 = gelu_erf(acc + bias)      (fc1)
  EPI_BIAS_RESID_F32 = 2,  // resid_f32 += acc + bias              (proj, fc2)
  EPI_BIAS_F32 = 3,        // out_f32 = acc + bias                 (generic / decoder)
  EPI_PATCH_F32 = 4,       // X[b, 1+i, :] = mix(acc + bias, mask_token) + pos[1+i]   (patch embedding)
  EPI_RESID_LN = 5,        // resid_f32 += acc + bias;  xn_bf16 = LayerNorm(resid_f32) * gamma + beta   (proj / fc2 + next LN)
  EPI_DGELU_BF16 = 6,      // out_bf16 = acc * gelu'(pre)          (training: input gradient of fc2 through the GELU, vit.py:59)
  EPI_RESID_SCALED_F32 = 7,  // resid_f32 += (acc + bias) * row_scale[row / rows_per_scale]   (proj, fc2 under stochastic depth;
                             // callers ask for it as EPI_BIAS_RESID_F32 with a row_scale, run_gemm picks this instantiation)
};

struct GemmArgs {
  int M, N;
  int kblocks;        // K / 64 per term
  int nterms;         // 1 (single 16-bit operands), 3 (split mode: hi*hi + hi*lo + lo*hi) or 2 (A split only: hi*hi + lo*hi)
  int lo_k;           // split mode: column where the lo halves of A and B start (= K)
  int a_lo_mask;      // bit t set: term t reads the lo half of A   (3 terms: 0b100, 2 terms: 0b10)
  int b_lo_mask;      // bit t set: term t reads the lo half of B   (3 terms: 0b010, 2 terms: 0)
  int gelu_mode;      // EPI_BIAS_GELU_BF16: 0 = three-coefficient sigmoid form (bf16 outputs), 1 = erff (fp32-parity mode),
                      // 2 = five-coefficient sigmoid form (fp16 outputs)
  int f16;            // 16-bit operand format of A, B and of bf16-typed outputs: 0 = bf16, 1 = IEEE fp16 (fp16 engines)
  const float* bias;  // [N] or nullptr
  int split_out;      // bf16 outputs only: 1 = also write lo = bf16(v - hi) at column offset lo_off;
                      // 2 (EPI_BIAS_GELU_BF16, training) = also write the pre-activation acc + bias at column offset lo_off
  int lo_off;
  // EPI_RESID_LN only: the LayerNorm that consumes the updated residual stream (vit.py:107/111), fused here
  const float* ln_gamma;
  const float* ln_beta;
  float ln_eps;
  __nv_bfloat16* xn;   // [M][ld_xn] bf16 normalised rows (A operand of the next GEMM)
  long long ld_xn;
  int num_clusters;    // persistent grid = num_clusters clusters of N / BN CTAs (one CTA per column block of a row tile)
  int debug;          // diagnostics only (VITOCM_GEMM_DEBUG): 1 = epilogue drains TMEM but skips math + stores, 2 = epilogue
                      // signals only (no TMEM load either)
  int stages;         // B_RES only: number of A stages that fit next to the resident B panel (host-computed)
  // A_PATCH / EPI_PATCH_F32 only
  const float* img;         // [B][C][H][W] fp32 pixels
  int img_h, img_w, patch;  // pixels; patch size p (multiple of 8)
  int n_patches;            // (H/p)*(W/p) per image
  const float* pos;         // [1 + n_patches][N] position table
  const float* mask;        // [B][n_patches] in {0,1} or nullptr (SimMIM mask-token mixing, SSS/model.py:31-33)
  const float* mask_token;  // [N]
  // A_PATCH, tile ingest straight from a gray uint8 mosaic (sliding_window + ToTensor, SSS/sw_processing.py:151-163, :236): image b of
  // this launch is window mos_t0 + b of the row-major grid mos_nx windows wide at stride mos_S, pixel value v / 255, zero beyond the mosaic; img is unused
  const uint8_t* mos;       // [mos_h][mos_pitch] or nullptr
  long long mos_pitch;
  int mos_h, mos_w, mos_nx, mos_S, mos_t0;
  float* out_f32;           // X [B][1 + n_patches][N] token stream
  int patch_tma;            // EPI_PATCH_F32: tmap_c = X as 2-D [B (1 + n_patches)][N] and tmap_d = pos [1 + n_patches][N] (fp32, 32 x 32 boxes,
                            // SWIZZLE_128B) are valid: position rows arrive and token rows leave through per-warp staging boxes
  // EPI_DGELU_BF16 only: the GELU's input saved by the forward fc1 epilogue, bf16 [M][ld_pre]
  const __nv_bfloat16* pre;
  long long ld_pre;
  // EPI_RESID_SCALED_F32 only: per-sample residual-branch scale (stochastic depth, vit.py:110-111), [M / rows_per_scale]
  const float* row_scale;
  int rows_per_scale;
  // PATCH_VAR only (images of different sizes packed back to back, no mask, no mosaic): vimg[b] = {patches before image b, patches per
  // row of image b, row of image b's CLS entry in the packed position tables pos, 0}, b < n_img, and vimg[n_img].x = M.  Image b's pixels
  // start at img + C p^2 vimg[b].x, its token rows at vimg[b].x + b of X; img_h, img_w and n_patches are unused.
  const int4* vimg;
  int n_img;
};

// PATCH_VAR: the image of patch row m (the last b with vimg[b].x <= m)
__device__ __forceinline__ int patch_image(const GemmArgs& a, int m) {
  int lo = 0, hi = a.n_img - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(&a.vimg[mid].x) <= m) lo = mid; else hi = mid - 1;
  }
  return lo;
}

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_EPI_WARP0 = 4;
// epilogue warps: 8 (two column halves per TMEM lane quadrant), or 12 with BN = 192 (three 64-column groups): the
// GELU epilogue is issue / latency bound, a third warp per scheduler hides its MUFU + FMA chains
__host__ __device__ constexpr int gemm_epi_warps(int BN, int EPI) { return ((EPI == 1 || EPI == 6) && BN == 192) ? 12 : 8; }
// patch embedding: 6 extra warps after the epilogue warps join warps 2-3 as A producers (8 producer warps)
constexpr int GEMM_PATCH_PRODUCER_WARPS = 8;
__host__ __device__ constexpr int gemm_threads(int BN, int EPI) {
  return (4 + gemm_epi_warps(BN, EPI) + (EPI == 4 ? GEMM_PATCH_PRODUCER_WARPS - 2 : 0)) * 32;
}
constexpr int GEMM_SMEM_LIMIT = 227 * 1024;

constexpr int GEMM_MAX_STAGES = 8;
constexpr int GEMM_PAIR_DEFAULT = 1;        // cta_group::2 for eligible shapes (VITOCM_GEMM_PAIR overrides)
constexpr int GEMM_RES_MAX_KBLOCKS = 6;     // B_RES: K <= 384

// B_RES ("weight panel resident"): for K <= 384 the whole [BN x K] weight panel stays in shared memory while the
// CTA walks down M (tiles are assigned n-major in contiguous ranges), so only A streams from L2.  The plain kernel
// re-fetches A and B for every tile: (128 + BN) * 128 B per 2*BN tensor clocks = 96-128 B/clk/SM, i.e. 14-19 KB/clk
// chip-wide against a measured L2->SM ceiling of ~9 KB/clk -- the GEMMs of this model were L2-bandwidth bound at
// 45-55 % of tensor peak.  With the panel resident the demand drops to 128*128 B per 2*BN clocks (43 B/clk at BN 192).
// EPI_RESID_LN ("fused LayerNorm"): a row of the residual stream spans CS = N / BN column tiles, owned by the CS CTAs
// of one thread-block cluster.  Every epilogue thread owns one row x 64 columns in registers, computes (mean, M2) of
// its 64 values exactly, writes the pair into the stats slab of every CTA of the cluster through distributed shared
// memory, and after a cluster-scope mbarrier round combines the (EPI_WARPS/4 * CS) partials with Chan's formula --
// full-row statistics without ever re-reading the row.  The separate LayerNorm kernel (one HBM pass over the fp32
// residual stream per LayerNorm) disappears.
// PAIR (cta_group::2): two CTAs of a cluster share one 256 x BN tile -- each stages its own 128 rows of A and only
// BN/2 rows of B per k-block, so the per-SM operand traffic drops from (128 + BN) to (128 + BN/2) rows per 2*BN
// tensor clocks (96 -> 64 B/clk/SM at BN = 256): the plain kernel is L2->SM bandwidth bound.
template <int BN, int EPI, bool B_RES = false, int CS = 1, bool PAIR = false>
struct GemmCfg {
  static constexpr bool OUT_BF16 = (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_GELU_BF16 || EPI == EPI_DGELU_BF16);
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;       // 16 KB
  static constexpr int B_BYTES = (PAIR ? BN / 2 : BN) * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + (B_RES ? 0 : B_BYTES);
  // per-warp epilogue staging: 2 x (32 x 32 fp32 box) or 2 x (32 x 32 bf16 box), double buffered; with a split
  // bf16 output the two bf16 boxes hold hi and lo instead (single buffered -- the parity mode is not the fast
  // path).  B_RES keeps one box per warp (single buffered) to leave room for the panel.
  static constexpr int STG_BOX_BYTES = OUT_BF16 ? 2048 : 4096;
  // LN: per warp two fp32 boxes (the residual rows come in and go out through them) + one bf16 box (normalised rows)
  // EPI_DGELU_BF16: a third bf16 box per warp receives the saved pre-activation tile by TMA
  static constexpr int STG_WARP_BYTES = EPI == EPI_RESID_LN ? 2 * 4096 + 2048 : (B_RES ? 1 : (EPI == EPI_DGELU_BF16 ? 3 : 2)) * STG_BOX_BYTES;
  static constexpr int EPI_WARPS = gemm_epi_warps(BN, EPI);
  static constexpr int STG_BYTES = EPI_WARPS * STG_WARP_BYTES;
  // EPI_RESID_LN: [2 slots][LN_SRC partial sources][128 rows] x (mean, M2)
  static constexpr int LN_SRC = (EPI_WARPS / 4) * CS;
  static constexpr int STATS_BYTES = EPI == EPI_RESID_LN ? 2 * LN_SRC * GEMM_BM * 8 : 0;
  static constexpr int FIXED_BYTES = STG_BYTES + STATS_BYTES + 1024 /*align slack*/ + 512 /*barriers*/;
  static constexpr int STAGES_FIT = (GEMM_SMEM_LIMIT - FIXED_BYTES) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_FIT > 6 ? 6 : STAGES_FIT;   // plain kernel (compile time)
  static constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + FIXED_BYTES;
  static_assert(B_RES || STAGES >= 3, "not enough shared memory for a 3-stage pipeline");
  // B_RES: stages next to a kblocks-deep panel
  static constexpr int res_stages(int kblocks) {
    const int fit = (GEMM_SMEM_LIMIT - FIXED_BYTES - kblocks * B_BYTES) / A_BYTES;
    return fit > GEMM_MAX_STAGES ? GEMM_MAX_STAGES : fit;
  }
  static constexpr int res_smem_bytes(int kblocks) { return res_stages(kblocks) * A_BYTES + kblocks * B_BYTES + FIXED_BYTES; }
};

// v / 255 for an 8-bit value, correctly rounded (== __fdiv_rn(v, 255.f), the ToTensor arithmetic) without the division: one
// residual-correction step on the reciprocal product is exact for all 256 inputs (checked exhaustively, tests/test_gpu_post.py)
__device__ __forceinline__ float u8_unit(uint32_t b) {
  constexpr float R = 1.0f / 255.0f;
  const float v = static_cast<float>(b);
  const float q = __fmul_rn(v, R);
  return __fmaf_rn(__fmaf_rn(-q, 255.0f, v), R, q);
}

// 8 consecutive A-tile values of the patch embedding -> one 16-byte shared-memory store: the hi part, or lo = v - hi, in the
// engine's 16-bit format (the format branch is warp uniform)
__device__ __forceinline__ void patch_store8(uint32_t addr, float (&v)[8], bool want_lo, bool f16) {
  if (f16) {
    if (want_lo) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] -= ptx::f16_round(v[j]);
    }
    ptx::sts_v4(addr, ptx::pack_f16x2(v[0], v[1]), ptx::pack_f16x2(v[2], v[3]), ptx::pack_f16x2(v[4], v[5]), ptx::pack_f16x2(v[6], v[7]));
  } else {
    if (want_lo) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] -= ptx::bf16_round(v[j]);
    }
    ptx::sts_v4(addr, ptx::pack_bf16x2(v[0], v[1]), ptx::pack_bf16x2(v[2], v[3]), ptx::pack_bf16x2(v[4], v[5]), ptx::pack_bf16x2(v[6], v[7]));
  }
}

__device__ __forceinline__ float gelu_erf(float x) {
  // nn.GELU() default (approximate='none'): x * Phi(x)
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// erf-GELU for two values at once on the packed-f32x2 pipe (bf16 mode; the output is rounded to bf16, 2^-9 relative):
//     gelu(x) = x * Phi(x),   Phi(x) ~= sigmoid(x * (a + b x^2 + c x^4))
// with (a, b, c) fitted to the exact Phi (erf form) over [-7, 7]: max |error| of gelu = 2.5e-5 (the familiar
// "tanh GELU" is the two-coefficient member of this family, 2.7e-4).  x^2 is clamped at 100 so the quintic stays
// monotone; sigmoid = rcp(1 + ex2(.)): 6 packed FMA-pipe instructions + 4 MUFU per pair, against 37 instructions per
// element for erff() -- the fc1 epilogue is issue bound, not tensor bound (K = 384 gives the tensor core only
// 0.09 clk of work per output element).  The fp32-parity mode keeps erff().
__device__ __forceinline__ void gelu_sigmoid_x2(float& x0, float& x1) {
  const uint64_t x2 = ptx::pack_f32x2(x0, x1);
  const uint64_t sq = ptx::mul_f32x2(x2, x2);
  float u0, u1;
  ptx::unpack_f32x2(sq, u0, u1);
  const uint64_t u = ptx::pack_f32x2(fminf(u0, 100.f), fminf(u1, 100.f));
  // coefficients pre-multiplied by -log2(e):  ex2(x * w) = exp(-x (a + b u + c u^2))
  uint64_t w = ptx::fma_f32x2(u, ptx::dup_f32x2(0.0010142630596f), ptx::dup_f32x2(-0.1067757240f));
  w = ptx::fma_f32x2(w, u, ptx::dup_f32x2(-2.3011213394f));
  const uint64_t arg = ptx::mul_f32x2(x2, w);
  float a0, a1;
  ptx::unpack_f32x2(arg, a0, a1);
  const uint64_t den = ptx::add_f32x2(ptx::pack_f32x2(ptx::ex2_approx(a0), ptx::ex2_approx(a1)), ptx::dup_f32x2(1.0f));
  float d0, d1;
  ptx::unpack_f32x2(den, d0, d1);
  const uint64_t r = ptx::mul_f32x2(x2, ptx::pack_f32x2(ptx::rcp_approx(d0), ptx::rcp_approx(d1)));
  ptx::unpack_f32x2(r, x0, x1);
}

// Five-coefficient member of the same family for fp16 engines (their outputs keep 11 significand bits, so the 2.5e-5 of the
// three-coefficient fit would show): Phi(x) ~= sigmoid(x (c0 + c1 u + c2 u^2 + c3 u^3 + c4 u^4)), u = min(x^2, 30), max |error|
// of gelu 3.0e-6 over [-8, 8] (fitted like the above; tests/test_gpu_kernels.py checks it against erf): two more FFMA2 per pair.
// No clamp of u in the code: the quartic keeps falling beyond u = 30 (w' < 0 there, the u^4 coefficient is negative), so the sigmoid only
// saturates harder -- gelu -> x or -> 0 as it should, through +-inf without a NaN (ex2(+inf) = inf, rcp(inf) = 0, x finite); the same
// 3.04e-6 maximum error with and without the clamp over [-12, 12], +-1e5 included.  Two FMNMX per pair fewer in an epilogue that is
// issue bound (the three-coefficient form above DOES need its clamp: its quadratic turns upwards at u = 53).
__device__ __forceinline__ void gelu_sigmoid5_x2(float& x0, float& x1) {
  const uint64_t x2 = ptx::pack_f32x2(x0, x1);
  const uint64_t u = ptx::mul_f32x2(x2, x2);
  // coefficients pre-multiplied by -log2(e)
  uint64_t w = ptx::fma_f32x2(u, ptx::dup_f32x2(-3.2290010e-06f), ptx::dup_f32x2(8.8238336e-05f));
  w = ptx::fma_f32x2(w, u, ptx::dup_f32x2(3.6027357e-04f));
  w = ptx::fma_f32x2(w, u, ptx::dup_f32x2(-0.10522669f));
  w = ptx::fma_f32x2(w, u, ptx::dup_f32x2(-2.3020453f));
  const uint64_t arg = ptx::mul_f32x2(x2, w);
  float a0, a1;
  ptx::unpack_f32x2(arg, a0, a1);
  const uint64_t den = ptx::add_f32x2(ptx::pack_f32x2(ptx::ex2_approx(a0), ptx::ex2_approx(a1)), ptx::dup_f32x2(1.0f));
  float d0, d1;
  ptx::unpack_f32x2(den, d0, d1);
  const uint64_t r = ptx::mul_f32x2(x2, ptx::pack_f32x2(ptx::rcp_approx(d0), ptx::rcp_approx(d1)));
  ptx::unpack_f32x2(r, x0, x1);
}

// Derivative of the same function, two values at once on the packed-f32x2 pipe:  gelu(x) = x * s(x),  s = sigmoid(t),
// t = x (a + b u + c u^2),  u = min(x^2, 100):
//     gelu'(x) = s + x s (1 - s) t'(x),   t' = a + 3 b u + 5 c u^2
// (beyond |x| = 10 the clamped u makes t' inexact, but s (1 - s) is 0 there in fp32).  Max |error| against the exact erf-form
// derivative 1.1e-4.  v <- v * gelu'(x): ~12 packed FMA-pipe instructions + 4 MUFU per pair -- scalar code made the
// input-gradient epilogue issue bound.
__device__ __forceinline__ void gelu_grad_mul_x2(float& v0, float& v1, float x0, float x1) {
  // (a, b, c) = -(coefficients of gelu_sigmoid_x2) / log2(e)
  constexpr float A = 1.595015768531f, B = 0.074011292043f, C = -0.000703033580f;
  const uint64_t x2 = ptx::pack_f32x2(x0, x1);
  const uint64_t sq = ptx::mul_f32x2(x2, x2);
  float u0, u1;
  ptx::unpack_f32x2(sq, u0, u1);
  const uint64_t u = ptx::pack_f32x2(fminf(u0, 100.f), fminf(u1, 100.f));
  const uint64_t poly = ptx::fma_f32x2(ptx::fma_f32x2(ptx::dup_f32x2(C), u, ptx::dup_f32x2(B)), u, ptx::dup_f32x2(A));
  const uint64_t arg = ptx::mul_f32x2(ptx::mul_f32x2(x2, poly), ptx::dup_f32x2(-1.4426950408889634f));
  float a0, a1;
  ptx::unpack_f32x2(arg, a0, a1);
  const uint64_t den = ptx::add_f32x2(ptx::pack_f32x2(ptx::ex2_approx(a0), ptx::ex2_approx(a1)), ptx::dup_f32x2(1.0f));
  float d0, d1;
  ptx::unpack_f32x2(den, d0, d1);
  const uint64_t sg = ptx::pack_f32x2(ptx::rcp_approx(d0), ptx::rcp_approx(d1));
  const uint64_t dt = ptx::fma_f32x2(ptx::fma_f32x2(ptx::dup_f32x2(5.0f * C), u, ptx::dup_f32x2(3.0f * B)), u, ptx::dup_f32x2(A));
  const uint64_t om = ptx::fma_f32x2(sg, ptx::dup_f32x2(-1.0f), ptx::dup_f32x2(1.0f));
  const uint64_t g = ptx::fma_f32x2(ptx::mul_f32x2(ptx::mul_f32x2(x2, sg), om), dt, sg);
  const uint64_t r = ptx::mul_f32x2(ptx::pack_f32x2(v0, v1), g);
  ptx::unpack_f32x2(r, v0, v1);
}

// Derivative of the five-coefficient form gelu_sigmoid5_x2 (fp16 engines, which run their forward fc1 in that form): with
// t = x P(u), P(u) = p0 + p1 u + p2 u^2 + p3 u^3 + p4 u^4 (= -(its coefficients) / log2(e)), u = x^2:
//     gelu'(x) = s + x s (1 - s) t'(x),   t' = p0 + 3 p1 u + 5 p2 u^2 + 7 p3 u^3 + 9 p4 u^4
// Max |error| against the exact erf-form derivative 1.5e-5 over [-12, 12].  No clamp of u: the saved input is fp16 (|x| <= 65504),
// where t' stays finite (< 1e35), and x s (1 - s) is exactly 0 once the sigmoid has saturated.  v <- v * gelu'(x).
__device__ __forceinline__ void gelu5_grad_mul_x2(float& v0, float& v1, float x0, float x1) {
  const uint64_t x2 = ptx::pack_f32x2(x0, x1);
  const uint64_t u = ptx::mul_f32x2(x2, x2);
  uint64_t poly = ptx::fma_f32x2(u, ptx::dup_f32x2(2.238172939e-06f), ptx::dup_f32x2(-6.116215382e-05f));
  poly = ptx::fma_f32x2(poly, u, ptx::dup_f32x2(-2.497226093e-04f));
  poly = ptx::fma_f32x2(poly, u, ptx::dup_f32x2(7.293758349e-02f));
  poly = ptx::fma_f32x2(poly, u, ptx::dup_f32x2(1.595656209f));
  const uint64_t arg = ptx::mul_f32x2(ptx::mul_f32x2(x2, poly), ptx::dup_f32x2(-1.4426950408889634f));
  float a0, a1;
  ptx::unpack_f32x2(arg, a0, a1);
  const uint64_t den = ptx::add_f32x2(ptx::pack_f32x2(ptx::ex2_approx(a0), ptx::ex2_approx(a1)), ptx::dup_f32x2(1.0f));
  float d0, d1;
  ptx::unpack_f32x2(den, d0, d1);
  const uint64_t sg = ptx::pack_f32x2(ptx::rcp_approx(d0), ptx::rcp_approx(d1));
  uint64_t dt = ptx::fma_f32x2(u, ptx::dup_f32x2(2.014355645e-05f), ptx::dup_f32x2(-4.281350767e-04f));
  dt = ptx::fma_f32x2(dt, u, ptx::dup_f32x2(-1.248613046e-03f));
  dt = ptx::fma_f32x2(dt, u, ptx::dup_f32x2(2.188127505e-01f));
  dt = ptx::fma_f32x2(dt, u, ptx::dup_f32x2(1.595656209f));
  const uint64_t om = ptx::fma_f32x2(sg, ptx::dup_f32x2(-1.0f), ptx::dup_f32x2(1.0f));
  const uint64_t g = ptx::fma_f32x2(ptx::mul_f32x2(ptx::mul_f32x2(x2, sg), om), dt, sg);
  const uint64_t r = ptx::mul_f32x2(ptx::pack_f32x2(v0, v1), g);
  ptx::unpack_f32x2(r, v0, v1);
}

// PATCH_VAR: patch embedding of images of different sizes (GemmArgs::vimg); A_PATCH and EPI_PATCH_F32 only
template <int BN, int EPI, bool A_PATCH, bool B_RES = false, int CS = 1, bool PAIR = false, bool PATCH_VAR = false>
__global__ void __launch_bounds__(gemm_threads(BN, EPI), 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                         const __grid_constant__ CUtensorMap tmap_c, const __grid_constant__ CUtensorMap tmap_d, const GemmArgs args) {
  using Cfg = GemmCfg<BN, EPI, B_RES, CS, PAIR>;
  constexpr bool LN = EPI == EPI_RESID_LN;
  static_assert(!(PAIR && (LN || A_PATCH || B_RES)), "cta_group::2 uses the plain pipeline and epilogues");
  constexpr int TILE_M = PAIR ? 2 * GEMM_BM : GEMM_BM;   // rows per tile (per CTA pair in PAIR mode)
  static_assert(LN || CS == 1, "clusters are only used by the fused-LayerNorm epilogue");
  static_assert(!(LN && (A_PATCH || B_RES)), "fused LayerNorm uses the plain pipeline");
  static_assert(!(A_PATCH && B_RES), "patch embedding uses the plain pipeline");
  static_assert(!PATCH_VAR || (A_PATCH && EPI == EPI_PATCH_F32), "PATCH_VAR is a patch-embedding mode");
  const int STAGES = B_RES ? args.stages : Cfg::STAGES;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment; all later accesses use 32-bit shared-window addresses
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_a = smem_base;
  const uint32_t smem_b = smem_base + STAGES * Cfg::A_BYTES;     // plain: [STAGES] B tiles; B_RES: the [kblocks] panel
  const uint32_t smem_stg = smem_b + (B_RES ? args.kblocks : STAGES) * Cfg::B_BYTES;
  const uint32_t smem_stats = smem_stg + Cfg::STG_BYTES;
  const uint32_t bars = smem_stats + Cfg::STATS_BYTES;
  const uint32_t full_bar = bars;                                   // [STAGES]  producers -> MMA
  const uint32_t empty_bar = bars + 8 * GEMM_MAX_STAGES;            // [STAGES]  MMA -> producers
  const uint32_t tfull_bar = bars + 16 * GEMM_MAX_STAGES;           // [2]       MMA -> epilogue
  const uint32_t tempty_bar = bars + 16 * GEMM_MAX_STAGES + 16;     // [2]       epilogue -> MMA
  const uint32_t bfull_bar = bars + 16 * GEMM_MAX_STAGES + 32;      // B_RES: panel loaded
  const uint32_t bempty_bar = bars + 16 * GEMM_MAX_STAGES + 40;     // B_RES: panel no longer read
  const uint32_t stat_bar = bars + 16 * GEMM_MAX_STAGES + 48;       // [2]  LN: partial statistics of a row tile arrived
  const uint32_t xin_bar = bars + 16 * GEMM_MAX_STAGES + 64;        // [12] per epilogue warp: residual boxes (LN) / pre-activation box (dGELU) landed
  const uint32_t tmem_ptr_smem = bars + 16 * GEMM_MAX_STAGES + 160;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_m = (args.M + TILE_M - 1) / TILE_M;
  const int tiles_n = args.N / BN;
  const int num_tiles = tiles_m * tiles_n;
  const int k_iters = args.kblocks * args.nterms;
  // tile schedule.  plain: m-major, strided over the persistent grid.  B_RES: n-major, one contiguous range per CTA
  // (so that a CTA changes weight panel at most a couple of times).
  // LN: cluster c walks row tiles c, c + num_clusters, ...; the CTA of rank r owns column tile r of each.
  const int cta_rank = (LN || PAIR) ? static_cast<int>(ptx::cluster_ctarank()) : 0;
  const int tile_begin = LN ? static_cast<int>(blockIdx.x) / CS
                            : PAIR ? static_cast<int>(blockIdx.x) / 2
                            : (B_RES ? static_cast<int>(static_cast<long long>(blockIdx.x) * num_tiles / gridDim.x) : static_cast<int>(blockIdx.x));
  const int tile_end = LN ? tiles_m : (B_RES ? static_cast<int>(static_cast<long long>(blockIdx.x + 1) * num_tiles / gridDim.x) : num_tiles);
  const int tile_step = LN ? args.num_clusters : PAIR ? static_cast<int>(gridDim.x) / 2 : (B_RES ? 1 : static_cast<int>(gridDim.x));
  const int pair_row = PAIR ? cta_rank * GEMM_BM : 0;   // this CTA's rows inside the 256-row pair tile
  auto tile_m = [&](int t) { return LN ? t : (B_RES ? t % tiles_m : t / tiles_n); };
  auto tile_n = [&](int t) { return LN ? cta_rank : (B_RES ? t / tiles_m : t % tiles_n); };

  if (warp == 0 && lane == 0) {
    if (!A_PATCH) ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_b);
    if (EPI != EPI_PATCH_F32) ptx::prefetch_tmap(&tmap_c);
    if (LN || EPI == EPI_DGELU_BF16) ptx::prefetch_tmap(&tmap_d);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(full_bar + 8 * s, A_PATCH ? 1 + GEMM_PATCH_PRODUCER_WARPS : 1);   // TMA thread (+ one arrive per A-producer warp)
      ptx::mbar_init(empty_bar + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(tfull_bar + 8 * s, 1);
      ptx::mbar_init(tempty_bar + 8 * s, Cfg::EPI_WARPS * (PAIR ? 2 : 1));  // one arrive per epilogue warp (of both CTAs)
    }
    ptx::mbar_init(bfull_bar, 1);
    ptx::mbar_init(bempty_bar, 1);
    ptx::mbar_init(stat_bar, 1);        // LN: one expect_tx arrive per row tile; the partials arrive as st.async complete_tx bytes
    ptx::mbar_init(stat_bar + 8, 1);
    for (int w = 0; w < 12; ++w) ptx::mbar_init(xin_bar + 8 * w, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    if (PAIR) {
      ptx::tmem_alloc_2cta(tmem_ptr_smem, Cfg::TMEM_COLS);
      ptx::tmem_relinquish_2cta();
    } else {
      ptx::tmem_alloc(tmem_ptr_smem, Cfg::TMEM_COLS);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if ((LN && CS > 1) || PAIR) ptx::cluster_sync_all();   // peers' barriers are initialised before anyone arrives on them remotely
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::lds_u32(tmem_ptr_smem);

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int cur_n = -1, panels = 0;
      for (int tile = tile_begin; tile < tile_end; tile += tile_step) {
        const int m0 = tile_m(tile) * TILE_M + pair_row;
        const int n0 = tile_n(tile) * BN + (PAIR ? cta_rank * (BN / 2) : 0);   // PAIR: this CTA stages its half of the B tile
        if (B_RES && tile_n(tile) != cur_n) {
          // (re)load the weight panel: kblocks boxes [BN x 64] -> smem_b, once the MMAs on the old panel retired
          if (panels > 0) ptx::mbar_wait(bempty_bar, (panels - 1) & 1, 6);
          ptx::mbar_arrive_expect_tx(bfull_bar, args.kblocks * Cfg::B_BYTES);
          for (int kb = 0; kb < args.kblocks; ++kb)
            ptx::tma_load_2d(smem_b + kb * Cfg::B_BYTES, &tmap_b, bfull_bar, kb * GEMM_BK, n0);
          cur_n = tile_n(tile);
          ++panels;
        }
        for (int it = 0; it < k_iters; ++it) {
          // operand order: term-major for TMA-fed A; k-block-major in patch mode so that the three terms of
          // one k-block re-read the same pixels out of L1
          const int term = A_PATCH ? it % args.nterms : it / args.kblocks;
          const int kb = A_PATCH ? it / args.nterms : it - term * args.kblocks;
          ptx::mbar_wait(empty_bar + 8 * stage, phase ^ 1, 1);
          // split mode terms: (hi,hi) (hi,lo) (lo,hi), or (hi,hi) (lo,hi) with a single-precision B; lo halves start at column K
          const int a_off = (((args.a_lo_mask >> term) & 1) ? args.lo_k : 0) + kb * GEMM_BK;
          const int b_off = (((args.b_lo_mask >> term) & 1) ? args.lo_k : 0) + kb * GEMM_BK;
          if (PAIR) {
            // both CTAs load into their own stage; all bytes complete on the leader's full barrier
            if (cta_rank == 0) ptx::mbar_arrive_expect_tx(full_bar + 8 * stage, 2 * Cfg::STAGE_BYTES);
            ptx::tma_load_2d_2cta(smem_a + stage * Cfg::A_BYTES, &tmap_a, full_bar + 8 * stage, a_off, m0);
            ptx::tma_load_2d_2cta(smem_b + stage * Cfg::B_BYTES, &tmap_b, full_bar + 8 * stage, b_off, n0);
          } else {
            ptx::mbar_arrive_expect_tx(full_bar + 8 * stage, A_PATCH ? Cfg::B_BYTES : Cfg::STAGE_BYTES);
            if (!A_PATCH) ptx::tma_load_2d(smem_a + stage * Cfg::A_BYTES, &tmap_a, full_bar + 8 * stage, a_off, m0);
            if (!B_RES) ptx::tma_load_2d(smem_b + stage * Cfg::B_BYTES, &tmap_b, full_bar + 8 * stage, b_off, n0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // One elected thread issues (elect.sync lets ptxas emit the tcgen05 instructions without a per-instruction
    // leader-election loop); descriptors are advanced by compile-time constants in fully unrolled loops.
    if ((!PAIR || cta_rank == 0) && ptx::elect_one()) {
      const uint32_t idesc = ptx::make_idesc(TILE_M, BN, false, false, args.f16 ? 0u : 1u);
      const uint64_t a_desc0 = ptx::make_smem_desc_sw128(smem_a, 1024, 0);
      const uint64_t b_desc0 = ptx::make_smem_desc_sw128(smem_b, 1024, 0);
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      int cur_n = -1, panels = 0;
      for (int tile = tile_begin; tile < tile_end; tile += tile_step) {
        if (B_RES && tile_n(tile) != cur_n) {
          ptx::mbar_wait(bfull_bar, panels & 1, 7);
          cur_n = tile_n(tile);
          ++panels;
        }
        ptx::mbar_wait(tempty_bar + 8 * as, aphase ^ 1, 2);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BN);
        for (int it = 0; it < k_iters; ++it) {
          ptx::mbar_wait(full_bar + 8 * stage, phase, 3);
          ptx::tc_fence_after();
          const uint64_t adesc = ptx::desc_advance(a_desc0, stage * Cfg::A_BYTES);
          const uint64_t bdesc = ptx::desc_advance(b_desc0, (B_RES ? it : stage) * Cfg::B_BYTES);
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            if (PAIR) ptx::umma_bf16_ss_2cta(d_tmem, ptx::desc_advance(adesc, k * 32), ptx::desc_advance(bdesc, k * 32), idesc, (it > 0 || k > 0) ? 1u : 0u);
            else ptx::umma_bf16_ss(d_tmem, ptx::desc_advance(adesc, k * 32), ptx::desc_advance(bdesc, k * 32), idesc, (it > 0 || k > 0) ? 1u : 0u);
          }
          // smem slot reusable once these MMAs retire (PAIR: in both CTAs)
          if (PAIR) ptx::umma_commit_2cta(empty_bar + 8 * stage); else ptx::umma_commit(empty_bar + 8 * stage);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        // accumulator complete (PAIR: each CTA's epilogue waits on its own copy of the barrier)
        if (PAIR) ptx::umma_commit_2cta(tfull_bar + 8 * as); else ptx::umma_commit(tfull_bar + 8 * as);
        if (B_RES && (tile + 1 >= tile_end || tile_n(tile + 1) != cur_n)) ptx::umma_commit(bempty_bar);  // panel free
        if (++as == 2) { as = 0; aphase ^= 1; }
      }
    }
  } else if (warp < GEMM_EPI_WARP0 || warp >= GEMM_EPI_WARP0 + Cfg::EPI_WARPS) {
    // ===================== A producer (patch embedding only) =====================
    // A[m, k] = bf16(x[b, c, py*p + yi, px*p + xi]),  m = b*n + py*Wp + px,  k = c*p*p + yi*p + xi.
    // One item = (row, 16-byte chunk): 8 consecutive pixels of one patch row -> 8 bf16 at the
    // SWIZZLE_128B position  row*128 + ((chunk ^ (row & 7)) << 4)  of the stage's A tile.
    if (A_PATCH) {
      // producer thread index 0..255: warps 2, 3 and the six warps after the epilogue warps
      const int t = (warp < GEMM_EPI_WARP0 ? warp - 2 : warp - (GEMM_EPI_WARP0 + Cfg::EPI_WARPS) + 2) * 32 + lane;
      const int p = args.patch, pp = p * p;
      const int Wp = args.img_w / p;
      const long long plane = static_cast<long long>(args.img_h) * args.img_w;
      const int chans = (args.kblocks * GEMM_BK) / pp;
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile_begin; tile < tile_end; tile += tile_step) {
        const int m0 = tile_m(tile) * GEMM_BM;
        for (int it = 0; it < k_iters; ++it) {
          const int term = it % args.nterms;
          const int kb = it / args.nterms;
          const bool want_lo = ((args.a_lo_mask >> term) & 1) != 0;
          ptx::mbar_wait(empty_bar + 8 * stage, phase ^ 1, 5);
          const uint32_t a_tile = smem_a + stage * Cfg::A_BYTES;
          // 4 items per thread: all 8 loads are issued before the first conversion so that their latencies overlap
          if (!PATCH_VAR && args.mos != nullptr) {   // gray uint8 mosaic: 8 pixels = 8 bytes of one mosaic row
            uint2 raw[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int item = t + 256 * u;
              const int chunk = item >> 7;
              const int row = item & 127;
              const int m = m0 + row;
              raw[u] = make_uint2(0u, 0u);
              if (m < args.M) {
                const int b = m / args.n_patches, i = m - b * args.n_patches;
                const int py = i / Wp, px = i - py * Wp;
                const int k = kb * GEMM_BK + chunk * 8;      // one channel: k = yi * p + xi
                const int yi = k / p, xi = k - yi * p;
                const int tl = args.mos_t0 + b;
                const int gy = (tl / args.mos_nx) * args.mos_S + py * p + yi;
                const int gx = (tl % args.mos_nx) * args.mos_S + px * p + xi;
                if (gy < args.mos_h && gx < args.mos_w) {
                  const uint8_t* src = args.mos + static_cast<long long>(gy) * args.mos_pitch + gx;
                  if (gx + 8 <= args.mos_w && (reinterpret_cast<uintptr_t>(src) & 7) == 0) {
                    raw[u] = __ldg(reinterpret_cast<const uint2*>(src));
                  } else {
                    unsigned long long acc = 0ull;
                    for (int j = 0; j < 8; ++j)
                      if (gx + j < args.mos_w) acc |= static_cast<unsigned long long>(__ldg(src + j)) << (8 * j);
                    raw[u] = make_uint2(static_cast<uint32_t>(acc), static_cast<uint32_t>(acc >> 32));
                  }
                }
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int item = t + 256 * u;
              const int chunk = item >> 7;
              const int row = item & 127;
              float v[8];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                v[j] = u8_unit((raw[u].x >> (8 * j)) & 0xffu);
                v[4 + j] = u8_unit((raw[u].y >> (8 * j)) & 0xffu);
              }
              patch_store8(a_tile + row * 128 + ((chunk ^ (row & 7)) << 4), v, want_lo, args.f16 != 0);
            }
          } else {
            float4 f[4][2];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int item = t + 256 * u;
              const int chunk = item >> 7;        // 0..7: consecutive threads -> consecutive rows (coalesced pixel reads)
              const int row = item & 127;
              const int m = m0 + row;
              f[u][0] = make_float4(0.f, 0.f, 0.f, 0.f);
              f[u][1] = f[u][0];
              if (m < args.M) {
                const float* src;
                if constexpr (PATCH_VAR) {
                  const int b = patch_image(args, m);
                  const int4 g = __ldg(args.vimg + b);
                  const int i = m - g.x, wpb = g.y, nb = __ldg(&args.vimg[b + 1].x) - g.x;
                  const int py = i / wpb, px = i - py * wpb;
                  const int k = kb * GEMM_BK + chunk * 8;
                  const int c = k / pp, rem = k - c * pp;
                  const int yi = rem / p, xi = rem - yi * p;
                  src = args.img + (static_cast<long long>(g.x) * chans + static_cast<long long>(c) * nb) * pp +
                        static_cast<long long>(py * p + yi) * (wpb * p) + px * p + xi;
                } else {
                const int b = m / args.n_patches, i = m - b * args.n_patches;
                const int py = i / Wp, px = i - py * Wp;
                const int k = kb * GEMM_BK + chunk * 8;
                const int c = k / pp, rem = k - c * pp;
                const int yi = rem / p, xi = rem - yi * p;
                src = args.img + (static_cast<long long>(b) * chans + c) * plane +
                                   static_cast<long long>(py * p + yi) * args.img_w + px * p + xi;
                }
                f[u][0] = __ldg(reinterpret_cast<const float4*>(src));
                f[u][1] = __ldg(reinterpret_cast<const float4*>(src) + 1);
              }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int item = t + 256 * u;
              const int chunk = item >> 7;
              const int row = item & 127;
              float v[8] = {f[u][0].x, f[u][0].y, f[u][0].z, f[u][0].w, f[u][1].x, f[u][1].y, f[u][1].z, f[u][1].w};
              patch_store8(a_tile + row * 128 + ((chunk ^ (row & 7)) << 4), v, want_lo, args.f16 != 0);
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(full_bar + 8 * stage);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue =====================
    const int q = warp & 3;                         // TMEM lane quadrant this warp may access
    const int ew = warp - GEMM_EPI_WARP0;           // 0..7
    const int half = ew >> 2;                       // which column group of the BN columns
    constexpr int COLS_PER_WARP = BN / (Cfg::EPI_WARPS / 4);
    const uint32_t stg_warp = smem_stg + ew * Cfg::STG_WARP_BYTES;
    const bool stg_single = B_RES || (Cfg::OUT_BF16 && args.split_out);   // one box, or both boxes used by one chunk (hi, lo)
    uint32_t stg_sel = 0;
    int as = 0;
    uint32_t aphase = 0;
    int ln_tiles = 0;
    uint32_t patch_phase = 0;   // EPI_PATCH_F32: phase of this warp's position-box barrier
    // EPI_DGELU_BF16: per-warp box for the saved pre-activation tile; the first request goes out before any accumulator is ready
    const uint32_t pre_box = stg_warp + 2 * Cfg::STG_BOX_BYTES;
    uint32_t pre_phase = 0;
    if (EPI == EPI_DGELU_BF16 && lane == 0 && tile_begin < tile_end) {
      ptx::mbar_arrive_expect_tx(xin_bar + 8 * ew, 2048);
      ptx::tma_load_2d(pre_box, &tmap_d, xin_bar + 8 * ew, tile_n(tile_begin) * BN + half * COLS_PER_WARP, tile_m(tile_begin) * TILE_M + pair_row + q * 32);
    }
    for (int tile = tile_begin; tile < tile_end; tile += tile_step) {
      const int m0 = tile_m(tile) * TILE_M + pair_row;
      const int n0 = tile_n(tile) * BN;
      const int row_base = m0 + q * 32;
      const int col_base = n0 + half * COLS_PER_WARP;
      if constexpr (LN) {
        static_assert(!LN || COLS_PER_WARP == 64, "fused LayerNorm: 64 columns per epilogue warp");
        constexpr int SRC = Cfg::LN_SRC;
        // staging of this warp: [box 0: cols 0..31 fp32][box 1: cols 32..63 fp32][bf16 box]
        const uint32_t xbox = stg_warp, nbox = stg_warp + 8192;
        const uint32_t my_xin = xin_bar + 8 * ew;
        // residual rows of this warp's 32 x 64 patch: two TMA boxes, fetched while the tile's MMAs are still running
        // (the boxes were last read by the previous tile's TMA stores)
        if (lane == 0) {
          ptx::bulk_wait_read0();
          ptx::mbar_arrive_expect_tx(my_xin, 8192);
          ptx::tma_load_2d(xbox, &tmap_c, my_xin, col_base, row_base);
          ptx::tma_load_2d(xbox + 4096, &tmap_c, my_xin, col_base + 32, row_base);
        }
        __syncwarp();
        ptx::mbar_wait(tfull_bar + 8 * as, aphase, 4);
        ptx::tc_fence_after();
        float y[2][32];
        uint32_t r0[32], r1[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * BN + half * COLS_PER_WARP), r0);
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * BN + half * COLS_PER_WARP + 32), r1);
        ptx::mbar_wait(my_xin, ln_tiles & 1, 9);
        ptx::tmem_ld_wait(r0);
        ptx::tmem_ld_wait(r1);
        // accumulator stage is in registers -> hand it back to the MMA warp right away
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(tempty_bar + 8 * as);
        if (++as == 2) { as = 0; aphase ^= 1; }
        float sum = 0.f;
        const int sw = lane & 7;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 xo = ptx::lds_v4f(xbox + g * 4096 + lane * 128 + ((j ^ sw) << 4));   // SWIZZLE_128B box row
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(args.bias + col_base + g * 32) + j);
            const uint32_t* rr = g == 0 ? r0 : r1;
            y[g][4 * j] = __uint_as_float(rr[4 * j]) + b4.x + xo.x;
            y[g][4 * j + 1] = __uint_as_float(rr[4 * j + 1]) + b4.y + xo.y;
            y[g][4 * j + 2] = __uint_as_float(rr[4 * j + 2]) + b4.z + xo.z;
            y[g][4 * j + 3] = __uint_as_float(rr[4 * j + 3]) + b4.w + xo.w;
            sum += (y[g][4 * j] + y[g][4 * j + 1]) + (y[g][4 * j + 2] + y[g][4 * j + 3]);
          }
        }
        // exact local statistics of the 64 values, published to every CTA of the cluster
        const float mean_i = sum * (1.0f / 64.0f);
        float m2_i = 0.f;
#pragma unroll
        for (int g = 0; g < 2; ++g)
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float d = y[g][j] - mean_i;
            m2_i = fmaf(d, d, m2_i);
          }
        const int slot = ln_tiles & 1;
        const uint32_t row_off = static_cast<uint32_t>((q * 32 + lane) * 8);
        const uint32_t mine = smem_stats + static_cast<uint32_t>(((slot * SRC + cta_rank * (Cfg::EPI_WARPS / 4) + half) * GEMM_BM) * 8) + row_off;
        // the first epilogue thread of the CTA announces how many bytes of partials this row tile will receive
        if (ew == 0 && lane == 0) ptx::mbar_arrive_expect_tx(stat_bar + 8 * slot, SRC * GEMM_BM * 8);
#pragma unroll
        for (int r = 0; r < CS; ++r) ptx::st_async_v2(ptx::mapa(mine, r), mean_i, m2_i, ptx::mapa(stat_bar + 8 * slot, r));
        // meanwhile: the updated residual rows go back out through the same boxes
#pragma unroll
        for (int g = 0; g < 2; ++g)
#pragma unroll
          for (int j = 0; j < 8; ++j)
            ptx::sts_v4(xbox + g * 4096 + lane * 128 + ((j ^ sw) << 4), __float_as_uint(y[g][4 * j]), __float_as_uint(y[g][4 * j + 1]),
                        __float_as_uint(y[g][4 * j + 2]), __float_as_uint(y[g][4 * j + 3]));
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_store_2d(&tmap_c, xbox, col_base, row_base);
          ptx::tma_store_2d(&tmap_c, xbox + 4096, col_base + 32, row_base);
          ptx::bulk_commit();
        }
        ptx::mbar_wait(stat_bar + 8 * slot, (ln_tiles >> 1) & 1, 8);
        ++ln_tiles;
        // Chan's combination of SRC groups of 64 values
        float mp[SRC];
        float mean = 0.f, m2 = 0.f;
#pragma unroll
        for (int p = 0; p < SRC; ++p) {
          const float2 v = ptx::lds_v2f(smem_stats + static_cast<uint32_t>(((slot * SRC + p) * GEMM_BM) * 8) + row_off);
          mp[p] = v.x;
          mean += v.x;
          m2 += v.y;
        }
        mean *= 1.0f / static_cast<float>(SRC);
#pragma unroll
        for (int p = 0; p < SRC; ++p) {
          const float d = mp[p] - mean;
          m2 = fmaf(64.0f * d, d, m2);
        }
        const float rstd = rsqrtf(m2 / static_cast<float>(args.N) + args.ln_eps);
        // normalised rows: bf16 box (32 x 32, SWIZZLE_64B) -> TMA store, one chunk at a time
        const int sw2 = (lane >> 1) & 3;
#pragma unroll
        for (int g = 0; g < 2; ++g) {
          const int col = col_base + g * 32;
          uint32_t pk[16];
          auto norm_pack = [&](auto f16_tag) {
            constexpr bool F16 = decltype(f16_tag)::value;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 g4 = __ldg(reinterpret_cast<const float4*>(args.ln_gamma + col) + j);
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(args.ln_beta + col) + j);
              pk[2 * j] = ptx::pack_h2<F16>((y[g][4 * j] - mean) * rstd * g4.x + b4.x, (y[g][4 * j + 1] - mean) * rstd * g4.y + b4.y);
              pk[2 * j + 1] = ptx::pack_h2<F16>((y[g][4 * j + 2] - mean) * rstd * g4.z + b4.z, (y[g][4 * j + 3] - mean) * rstd * g4.w + b4.w);
            }
          };
          if (args.f16) norm_pack(std::true_type{}); else norm_pack(std::false_type{});
          if (g == 1) {   // the bf16 box is still being read by the first chunk's store
            if (lane == 0) ptx::bulk_wait_read0();
            __syncwarp();
          }
#pragma unroll
          for (int j = 0; j < 4; ++j)
            ptx::sts_v4(nbox + lane * 64 + ((j ^ sw2) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_2d(&tmap_d, nbox, col, row_base);
            ptx::bulk_commit();
          }
        }
        continue;
      }
      ptx::mbar_wait(tfull_bar + 8 * as, aphase, 4);
      ptx::tc_fence_after();
      if (args.debug == 3) {   // diagnostics: drain the warp's slice with back-to-back loads and one wait
        constexpr int NCH = COLS_PER_WARP / 32;
        uint32_t rr[NCH][32];
#pragma unroll
        for (int g = 0; g < NCH; ++g)
          ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * BN + half * COLS_PER_WARP + g * 32), rr[g]);
#pragma unroll
        for (int g = 0; g < NCH; ++g) ptx::tmem_ld_wait(rr[g]);
        uint32_t acc = 0;
#pragma unroll
        for (int g = 0; g < NCH; ++g)
#pragma unroll
          for (int j = 0; j < 32; ++j) acc ^= rr[g][j];
        if (acc == 0x7fc12345u) args.out_f32[0] = 1.f;
      }
#pragma unroll 1
      for (int c = 0; c < COLS_PER_WARP; c += 32) {
        const int col = col_base + c;
        if (args.debug >= 2) continue;
        // EPI_PATCH_F32, staged path: the 32 patch rows of this warp lie inside one image (and inside M), so their position rows
        // and their token rows are 32 consecutive rows of pos / X: one TMA box in, one out.  (Each lane writing its own 128 bytes
        // cost 32 partial sectors per store instruction: the kernel ran 6 x above its HBM floor.)  Warps that straddle an image
        // boundary -- one in ~49 -- keep the per-lane path.
        bool patch_fast = false;
        int patch_i0 = 0, patch_b0 = 0;
        int patch_pos0 = 0, patch_tok0 = 0;   // PATCH_VAR: first position / token row of the warp's image
        if constexpr (PATCH_VAR) {   // (a warp's 32 rows inside one image: one position box in, one token box out, as below)
          patch_b0 = patch_image(args, row_base < args.M ? row_base : args.M - 1);
          const int4 g = __ldg(args.vimg + patch_b0);
          patch_i0 = row_base - g.x;
          patch_pos0 = g.z;
          patch_tok0 = g.x + patch_b0;
          patch_fast = args.patch_tma != 0 && row_base + 32 <= args.M && g.x + patch_i0 + 32 <= __ldg(&args.vimg[patch_b0 + 1].x);
          if (patch_fast && lane == 0) {
            ptx::mbar_arrive_expect_tx(xin_bar + 8 * ew, 4096);
            ptx::tma_load_2d(stg_warp, &tmap_d, xin_bar + 8 * ew, col, patch_pos0 + 1 + patch_i0);
          }
        } else if (EPI == EPI_PATCH_F32) {
          patch_b0 = row_base / args.n_patches;
          patch_i0 = row_base - patch_b0 * args.n_patches;
          patch_fast = args.patch_tma != 0 && row_base + 32 <= args.M && patch_i0 + 32 <= args.n_patches;
          if (patch_fast && lane == 0) {   // the box was last read (synchronously) by this warp's previous chunk
            ptx::mbar_arrive_expect_tx(xin_bar + 8 * ew, 4096);
            ptx::tma_load_2d(stg_warp, &tmap_d, xin_bar + 8 * ew, col, 1 + patch_i0);
          }
        }
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * BN + half * COLS_PER_WARP + c), r);
        float bv[32];
        if (args.bias != nullptr) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(args.bias + col) + j);   // same address in every lane
            bv[4 * j] = b4.x; bv[4 * j + 1] = b4.y; bv[4 * j + 2] = b4.z; bv[4 * j + 3] = b4.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) bv[j] = 0.f;
        }
        ptx::tmem_ld_wait(r);
        uint4 pq[4];   // EPI_DGELU_BF16: this lane's 32 saved GELU inputs out of the TMA-staged box (32 rows x 64 B, SWIZZLE_64B)
        if (EPI == EPI_DGELU_BF16) {
          ptx::mbar_wait(xin_bar + 8 * ew, pre_phase, 9);
          pre_phase ^= 1u;
          const uint32_t prow = pre_box + lane * 64;
          const int psw = (lane >> 1) & 3;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const float4 f = ptx::lds_v4f(prow + ((g ^ psw) << 4));
            pq[g] = make_uint4(__float_as_uint(f.x), __float_as_uint(f.y), __float_as_uint(f.z), __float_as_uint(f.w));
          }
          // the box is in registers: request the next one (this tile's next chunk, or the next tile's first) so that its
          // latency hides under this chunk's math and store
          __syncwarp();
          int nt = tile, nc = c + 32;
          if (nc >= COLS_PER_WARP) { nt = tile + tile_step; nc = 0; }
          if (lane == 0 && nt < tile_end) {
            ptx::mbar_arrive_expect_tx(xin_bar + 8 * ew, 2048);
            ptx::tma_load_2d(pre_box, &tmap_d, xin_bar + 8 * ew, tile_n(nt) * BN + half * COLS_PER_WARP + nc, tile_m(nt) * TILE_M + pair_row + q * 32);
          }
        }
        if (args.debug == 1) {
          uint32_t acc = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j) acc ^= r[j];
          if (acc == 0x7fc12345u) args.out_f32[0] = 1.f;   // keep the load alive
          continue;
        }
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]) + bv[j];
        if (EPI == EPI_DGELU_BF16) {   // the derivative of the GELU form the forward used: gelu_mode 2 on fp16 engines, else 0
          if (args.f16) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const uint32_t wds[4] = {pq[g].x, pq[g].y, pq[g].z, pq[g].w};
#pragma unroll
              for (int k = 0; k < 4; ++k)
                gelu5_grad_mul_x2(v[8 * g + 2 * k], v[8 * g + 2 * k + 1], __half2float(__ushort_as_half(static_cast<unsigned short>(wds[k] & 0xffffu))),
                                  __half2float(__ushort_as_half(static_cast<unsigned short>(wds[k] >> 16))));
            }
          } else {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              const uint32_t wds[4] = {pq[g].x, pq[g].y, pq[g].z, pq[g].w};
#pragma unroll
              for (int k = 0; k < 4; ++k)
                gelu_grad_mul_x2(v[8 * g + 2 * k], v[8 * g + 2 * k + 1], __uint_as_float(wds[k] << 16), __uint_as_float(wds[k] & 0xffff0000u));
            }
          }
        }
        uint32_t pre[16];   // training: the GELU input, kept for the backward (vit.py:59), in the engine's 16-bit format
        if (EPI == EPI_BIAS_GELU_BF16 && args.split_out == 2) {
          if (args.f16) {
#pragma unroll
            for (int j = 0; j < 16; ++j) pre[j] = ptx::pack_f16x2(v[2 * j], v[2 * j + 1]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) pre[j] = ptx::pack_bf16x2(v[2 * j], v[2 * j + 1]);
          }
        }
        if (EPI == EPI_BIAS_GELU_BF16) {
          if (args.gelu_mode == 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 2) gelu_sigmoid_x2(v[j], v[j + 1]);
          } else if (args.gelu_mode == 2) {
#pragma unroll
            for (int j = 0; j < 32; j += 2) gelu_sigmoid5_x2(v[j], v[j + 1]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
          }
        }
        if (EPI == EPI_PATCH_F32) {
          // token row of patch m = b*n + i is b*(n+1) + 1 + i: the row remap (and the +1 jump at image
          // boundaries inside a chunk) rules out a box store; each lane writes its own 128 contiguous bytes
          const int m = row_base + lane;
          if (patch_fast) {
            if (args.mask != nullptr) {
              const float mk = __ldg(args.mask + m);
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = v[j] * (1.f - mk) + __ldg(args.mask_token + col + j) * mk;
            }
            const uint32_t posbox = stg_warp + lane * 128, outbox = stg_warp + 4096 + lane * 128;
            const int sw = lane & 7;
            ptx::mbar_wait(xin_bar + 8 * ew, patch_phase, 10);
            patch_phase ^= 1u;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 p4 = ptx::lds_v4f(posbox + ((j ^ sw) << 4));
              v[4 * j] += p4.x; v[4 * j + 1] += p4.y; v[4 * j + 2] += p4.z; v[4 * j + 3] += p4.w;
            }
            if (lane == 0) ptx::bulk_wait_read0();   // the previous token box has been read by its store
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; ++j)
              ptx::sts_v4(outbox + ((j ^ sw) << 4), __float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                          __float_as_uint(v[4 * j + 3]));
            ptx::fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
              ptx::tma_store_2d(&tmap_c, stg_warp + 4096, col, PATCH_VAR ? patch_tok0 + 1 + patch_i0 : patch_b0 * (args.n_patches + 1) + 1 + patch_i0);
              ptx::bulk_commit();
            }
            continue;
          }
          if (PATCH_VAR && m < args.M) {
            const int b = patch_image(args, m);
            const int4 g = __ldg(args.vimg + b);
            const int i = m - g.x;
            const float4* pr = reinterpret_cast<const float4*>(args.pos + static_cast<long long>(g.z + 1 + i) * args.N + col);
            float4* orow = reinterpret_cast<float4*>(args.out_f32 + static_cast<long long>(g.x + b + 1 + i) * args.N + col);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 p4 = __ldg(pr + j);
              orow[j] = make_float4(v[4 * j] + p4.x, v[4 * j + 1] + p4.y, v[4 * j + 2] + p4.z, v[4 * j + 3] + p4.w);
            }
          } else if (m < args.M) {
            const int b = m / args.n_patches, i = m - b * args.n_patches;
            if (args.mask != nullptr) {
              const float mk = __ldg(args.mask + m);
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = v[j] * (1.f - mk) + __ldg(args.mask_token + col + j) * mk;
            }
            const float4* pr = reinterpret_cast<const float4*>(args.pos + static_cast<long long>(1 + i) * args.N + col);
            float4* orow = reinterpret_cast<float4*>(args.out_f32 + (static_cast<long long>(b) * (args.n_patches + 1) + 1 + i) * args.N + col);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 p4 = __ldg(pr + j);
              orow[j] = make_float4(v[4 * j] + p4.x, v[4 * j + 1] + p4.y, v[4 * j + 2] + p4.z, v[4 * j + 3] + p4.w);
            }
          }
          continue;
        }
        // the TMA store that last used this staging box must have finished reading it
        const uint32_t stg = stg_warp + (stg_single ? 0u : stg_sel * Cfg::STG_BOX_BYTES);
        stg_sel ^= 1u;
        if (lane == 0) {
          if (stg_single) ptx::bulk_wait_read0(); else ptx::bulk_wait_read1();
        }
        __syncwarp();
        if (Cfg::OUT_BF16) {
          // 32 rows x 64 B, SWIZZLE_64B: 16-byte chunk j of row r sits at r*64 + ((j ^ ((r >> 1) & 3)) << 4)
          const uint32_t rowaddr = stg + lane * 64;
          const int sw = (lane >> 1) & 3;
          auto put_rows = [&](auto f16_tag) {   // hi (and lo = v - hi) in the engine's 16-bit format; the format branch is warp uniform
            constexpr bool F16 = decltype(f16_tag)::value;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              ptx::sts_v4(rowaddr + ((j ^ sw) << 4), ptx::pack_h2<F16>(v[8 * j], v[8 * j + 1]), ptx::pack_h2<F16>(v[8 * j + 2], v[8 * j + 3]),
                          ptx::pack_h2<F16>(v[8 * j + 4], v[8 * j + 5]), ptx::pack_h2<F16>(v[8 * j + 6], v[8 * j + 7]));
            if (EPI == EPI_BIAS_GELU_BF16 && args.split_out == 2) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                ptx::sts_v4(rowaddr + Cfg::STG_BOX_BYTES + ((j ^ sw) << 4), pre[4 * j], pre[4 * j + 1], pre[4 * j + 2], pre[4 * j + 3]);
            } else if (args.split_out) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] -= ptx::round_h<F16>(v[j]);
#pragma unroll
              for (int j = 0; j < 4; ++j)
                ptx::sts_v4(rowaddr + Cfg::STG_BOX_BYTES + ((j ^ sw) << 4), ptx::pack_h2<F16>(v[8 * j], v[8 * j + 1]), ptx::pack_h2<F16>(v[8 * j + 2], v[8 * j + 3]),
                            ptx::pack_h2<F16>(v[8 * j + 4], v[8 * j + 5]), ptx::pack_h2<F16>(v[8 * j + 6], v[8 * j + 7]));
            }
          };
          if (args.f16) put_rows(std::true_type{}); else put_rows(std::false_type{});
        } else {
          if (EPI == EPI_RESID_SCALED_F32) {   // one load per row; rows past M are clipped by the TMA
            const int m = row_base + lane;
            const float s = m < args.M ? __ldg(args.row_scale + m / args.rows_per_scale) : 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= s;
          }
          // 32 rows x 128 B, SWIZZLE_128B: chunk j of row r sits at r*128 + ((j ^ (r & 7)) << 4)
          const uint32_t rowaddr = stg + lane * 128;
          const int sw = lane & 7;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            ptx::sts_v4(rowaddr + ((j ^ sw) << 4), __float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                        __float_as_uint(v[4 * j + 3]));
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (EPI == EPI_BIAS_RESID_F32 || EPI == EPI_RESID_SCALED_F32) {
            ptx::tma_reduce_add_2d(&tmap_c, stg, col, row_base);
          } else {
            ptx::tma_store_2d(&tmap_c, stg, col, row_base);
            if (Cfg::OUT_BF16 && args.split_out) ptx::tma_store_2d(&tmap_c, stg + Cfg::STG_BOX_BYTES, col + args.lo_off, row_base);
          }
          ptx::bulk_commit();
        }
      }
      // accumulator stage fully read into registers -> hand it back to the MMA warp (PAIR: the leader CTA's)
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) ptx::mbar_arrive_leader(tempty_bar + 8 * as); else ptx::mbar_arrive(tempty_bar + 8 * as);
      }
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
    if (lane == 0) ptx::bulk_wait_all0();   // global writes complete before the CTA exits
  }

  ptx::tc_fence_before();
  __syncthreads();
  if ((LN && CS > 1) || PAIR) ptx::cluster_sync_all();   // no CTA leaves while a peer could still address its shared memory / TMEM
  if (warp == 2) {
    ptx::tc_fence_after();
    if (PAIR) ptx::tmem_dealloc_2cta(tmem_base, Cfg::TMEM_COLS); else ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace vitocm
