// Weight-gradient GEMM for sm_100a (training step of SSS/mim.py:153-182, the `loss.backward()` half of every
// nn.Linear on the path: vit.py:58,61,80,88, the patch-embedding conv vit.py:127 and the MIM decoder model.py:61-64):
//     dW[R, C] += sum_m G[m, R]^T * A[m, C]          (G = dL/dY, A = the layer's input, both bf16 row-major [M, ld])
// The contraction runs over the TOKEN axis, i.e. over the rows of both operands, so both are "MN-major" for the
// tensor core: a TMA box of [64 tokens] x [64 features] (128-byte rows, SWIZZLE_128B) is exactly one MN-major
// core-matrix atom (8-token groups 1024 B apart = SBO, 64-feature atoms LBO apart).  No transposed copy of any
// activation is ever written to HBM.
//
// Work item = (128-row tile of dW, NB x BN column tile, token split).  One CTA per item: warp 0 = TMA producer,
// warp 1 = MMA issuer (one elected thread) + TMEM allocator, warps 2..5 = epilogue.  The accumulator
// (128 x NB*BN fp32) lives in TMEM for the whole token range; the epilogue adds it into the fp32 gradient with
// TMA reduce-add (cp.reduce.async.bulk.tensor .add, performed by the L2), which is also how token splits combine.
// Bias gradient for free: the column sums of G are G^T . 1, so the CTAs of the first column tile issue one extra N = 16 MMA per
// k-step against a constant all-ones B tile (8 KB of bf16 1.0: any swizzle of ones is ones) into 16 spare TMEM columns; the
// epilogue adds column 0 into db with 128 atomics per CTA.  No separate pass over G.
// F16 = true: fp16 operands (fp16 engines).  G then carries the loss scale S of the training step, and the epilogue multiplies
// the accumulator (and the bias column) by *inv_scale = 1 / S before the reduce-add: exact, S being a power of two.
#pragma once
#include "ptx.cuh"

namespace vitocm {

struct WgradArgs {
  int M;          // tokens (rows of G and A)
  int R, C;       // dW is [R][C]
  int tiles_c;    // C tiles of NB*BN columns
  int splits;     // token splits
  int kblocks;    // ceil(M / 64)
  float* colsum;  // [R] or nullptr: colsum[r] += sum_m G[m][r] -- the bias gradient of the same Linear, from the tensor core
  const float* inv_scale;   // F16 only: device scalar multiplied into dW and colsum (nullptr: 1)
};

constexpr int WG_BM = 128;      // rows of dW per tile (features of G)
constexpr int WG_BKT = 64;      // tokens per pipeline stage
constexpr int WG_THREADS = 192;
constexpr int WG_ATOM_BYTES = WG_BKT * 128;   // [64 tokens][64 bf16]

template <int BN, int NB>
struct WgradCfg {
  static constexpr int WIDTH = BN * NB;
  static constexpr int A_BYTES = 2 * WG_ATOM_BYTES;                 // 128 features of G
  static constexpr int B_BYTES = (WIDTH / 64) * WG_ATOM_BYTES;      // WIDTH features of A
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STG_BYTES = 4 * 4096;                        // per epilogue warp one 32 x 32 fp32 box
  static constexpr int ONES_BYTES = WG_ATOM_BYTES;                  // [64 tokens][64 x 16-bit 1.0]
  static constexpr int FIXED = STG_BYTES + ONES_BYTES + 1024 + 256;
  static constexpr int STAGES_FIT = (227 * 1024 - FIXED) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_FIT > 6 ? 6 : STAGES_FIT;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + FIXED;
  static constexpr int ACC_COLS = WIDTH + 16;                       // + the bias-gradient accumulator
  static constexpr int TMEM_COLS = ACC_COLS <= 32 ? 32 : ACC_COLS <= 64 ? 64 : ACC_COLS <= 128 ? 128 : ACC_COLS <= 256 ? 256 : 512;
  static_assert(BN % 64 == 0 && BN <= 256 && ACC_COLS <= 512, "tile width");
  static_assert(STAGES >= 3, "not enough shared memory for a 3-stage pipeline");
};

template <int BN, int NB, bool F16 = false>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_g, const __grid_constant__ CUtensorMap tmap_a,
                          const __grid_constant__ CUtensorMap tmap_w, const WgradArgs args) {
  using Cfg = WgradCfg<BN, NB>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_stg = smem_base + STAGES * Cfg::STAGE_BYTES;
  const uint32_t smem_ones = smem_stg + Cfg::STG_BYTES;
  const uint32_t bars = smem_ones + Cfg::ONES_BYTES;
  const uint32_t full_bar = bars;              // [STAGES]
  const uint32_t empty_bar = bars + 64;        // [STAGES]
  const uint32_t acc_bar = bars + 128;         // accumulator complete
  const uint32_t tmem_ptr_smem = bars + 136;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // work item
  int item = blockIdx.x;
  const int split = item % args.splits; item /= args.splits;
  const int tc = item % args.tiles_c;
  const int tr = item / args.tiles_c;
  const int r0 = tr * WG_BM, c0 = tc * Cfg::WIDTH;
  const int kb0 = static_cast<int>(static_cast<long long>(split) * args.kblocks / args.splits);
  const int kb1 = static_cast<int>(static_cast<long long>(split + 1) * args.kblocks / args.splits);
  const int nk = kb1 - kb0;
  const bool do_colsum = args.colsum != nullptr && tc == 0;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_g);
    ptx::prefetch_tmap(&tmap_a);
    ptx::prefetch_tmap(&tmap_w);
    for (int s = 0; s < STAGES; ++s) {
      ptx::mbar_init(full_bar + 8 * s, 1);
      ptx::mbar_init(empty_bar + 8 * s, 1);
    }
    ptx::mbar_init(acc_bar, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(tmem_ptr_smem, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  if (do_colsum && warp >= 2) {   // the all-ones B tile of the bias-gradient MMA
    constexpr uint32_t ONE2 = F16 ? 0x3c003c00u : 0x3f803f80u;   // 1.0 twice, fp16 / bf16
    for (int i = (warp - 2) * 32 + lane; i < Cfg::ONES_BYTES / 16; i += 128)
      ptx::sts_v4(smem_ones + i * 16, ONE2, ONE2, ONE2, ONE2);
    ptx::fence_proxy_async_smem();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::lds_u32(tmem_ptr_smem);

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nk; ++it) {
        const int m0 = (kb0 + it) * WG_BKT;
        ptx::mbar_wait(empty_bar + 8 * stage, phase ^ 1, 31);
        ptx::mbar_arrive_expect_tx(full_bar + 8 * stage, Cfg::STAGE_BYTES);
        const uint32_t a_tile = smem_base + stage * Cfg::STAGE_BYTES;
        const uint32_t b_tile = a_tile + Cfg::A_BYTES;
#pragma unroll
        for (int a = 0; a < 2; ++a) ptx::tma_load_2d(a_tile + a * WG_ATOM_BYTES, &tmap_g, full_bar + 8 * stage, r0 + 64 * a, m0);
#pragma unroll
        for (int b = 0; b < Cfg::WIDTH / 64; ++b) ptx::tma_load_2d(b_tile + b * WG_ATOM_BYTES, &tmap_a, full_bar + 8 * stage, c0 + 64 * b, m0);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      constexpr uint32_t idesc = ptx::make_idesc(WG_BM, BN, /*A MN-major*/ true, /*B MN-major*/ true, F16 ? 0u : 1u);
      constexpr uint32_t idesc_ones = ptx::make_idesc(WG_BM, 16, true, true, F16 ? 0u : 1u);
      const uint64_t ones_desc = ptx::make_smem_desc_sw128(smem_ones, 1024, WG_ATOM_BYTES);
      int stage = 0;
      uint32_t phase = 0;
      for (int it = 0; it < nk; ++it) {
        ptx::mbar_wait(full_bar + 8 * stage, phase, 32);
        ptx::tc_fence_after();
        const uint32_t a_tile = smem_base + stage * Cfg::STAGE_BYTES;
        // MN-major SWIZZLE_128B: 8-token groups 1024 B apart (SBO), 64-feature atoms WG_ATOM_BYTES apart (LBO);
        // one MMA consumes 16 tokens = 2048 B of every atom
        const uint64_t adesc = ptx::make_smem_desc_sw128(a_tile, 1024, WG_ATOM_BYTES);
        const uint64_t bdesc = ptx::make_smem_desc_sw128(a_tile + Cfg::A_BYTES, 1024, WG_ATOM_BYTES);
#pragma unroll
        for (int k = 0; k < WG_BKT / 16; ++k) {
#pragma unroll
          for (int nb = 0; nb < NB; ++nb)
            ptx::umma_bf16_ss(tmem_base + nb * BN, ptx::desc_advance(adesc, k * 2048),
                              ptx::desc_advance(bdesc, nb * (BN / 64) * WG_ATOM_BYTES + k * 2048), idesc, (it > 0 || k > 0) ? 1u : 0u);
          if (do_colsum)
            ptx::umma_bf16_ss(tmem_base + Cfg::WIDTH, ptx::desc_advance(adesc, k * 2048), ptx::desc_advance(ones_desc, k * 2048), idesc_ones,
                              (it > 0 || k > 0) ? 1u : 0u);
        }
        ptx::umma_commit(empty_bar + 8 * stage);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      ptx::umma_commit(acc_bar);
    }
  } else if (nk > 0) {
    // ===================== epilogue: dW tile += accumulator =====================
    const int q = warp & 3;   // TMEM lane quadrant of this warp (warps 2..5 -> 2, 3, 0, 1)
    const uint32_t stg = smem_stg + q * 4096;
    ptx::mbar_wait(acc_bar, 0, 33);
    ptx::tc_fence_after();
    const int row = r0 + q * 32;
    const float inv = F16 && args.inv_scale != nullptr ? *args.inv_scale : 1.0f;
    if (do_colsum) {   // column 0 of the ones-MMA accumulator = sum over this split's tokens of G[:, row + lane]
      uint32_t cs;
      ptx::tmem_ld_32x32b_x1(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(Cfg::WIDTH), cs);
      ptx::tmem_ld_wait1(cs);
      if (row + lane < args.R) atomicAdd(args.colsum + row + lane, F16 ? __uint_as_float(cs) * inv : __uint_as_float(cs));
    }
    if (row < args.R) {
#pragma unroll 1
      for (int c = 0; c < Cfg::WIDTH; c += 32) {
        if (c0 + c >= args.C) break;
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(c), r);
        if (lane == 0) ptx::bulk_wait_read0();   // the previous chunk's reduce has finished reading the box
        __syncwarp();
        ptx::tmem_ld_wait(r);
        if (F16) {
#pragma unroll
          for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) * inv);
        }
        const uint32_t rowaddr = stg + lane * 128;
        const int sw = lane & 7;
#pragma unroll
        for (int j = 0; j < 8; ++j) ptx::sts_v4(rowaddr + ((j ^ sw) << 4), r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          ptx::tma_reduce_add_2d(&tmap_w, stg, c0 + c, row);
          ptx::bulk_commit();
        }
      }
    }
    if (lane == 0) ptx::bulk_wait_all0();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace vitocm
