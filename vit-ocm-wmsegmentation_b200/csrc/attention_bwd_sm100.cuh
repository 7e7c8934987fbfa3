// Flash-attention backward for sm_100a (head_dim DH = 64 or 128), tcgen05 + TMEM + TMA -- the `loss.backward()` half of
// SSS/dino/vision_transformer.py:83-87 (q@k^T*scale, softmax, attn@v) inside the MIM training step (SSS/mim.py:153-182).
// Nothing N x N is ever written to HBM: P is recomputed from the saved log-sum-exp of the forward pass.
//
//   given  dO = dL/dctx,  LSE2[q] = log2 sum_k exp(scale * q.k)  (forward),  Delta[q] = sum_d dO[q,d] * O[q,d]:
//     P   = exp2(scale*log2e * Q K^T - LSE2)                 dV = P^T dO
//     dP  = dO V^T                                           dK = dS^T Q
//     dS  = scale * P o (dP - Delta)                         dQ = dS K
//
// One work item = one (image b, head h, 128-key block j): K_j, V_j stay in shared memory, dK_j, dV_j accumulate in TMEM
// over the 128-query tiles i.  CTAs are persistent (one per SM) and walk the items: barrier phases, the Q/dO ring, the
// double-buffered K/V slot and TMEM live across items, so the next item's K/V arrive under the current item's last tiles
// and its first S / dP MMAs run while dK_j / dV_j are drained.  Per (i, j):
//   MMA   S  = Q_i K_j^T, dP = dO_i V_j^T                    (K-major operands)            -> TMEM S | dP
//   warps 0..3 (thread = query row): tcgen05.ld S, dP -> P, dS (16-bit) -> shared memory, row-major [q][k]
//   MMA   dV += P^T dO_i, dK += dS^T Q_i                     (A = P / dS read MN-major: the contraction runs over the
//                                                             rows q; B = dO_i / Q_i MN-major)  -> TMEM dV | dK
//   MMA   dQ_i = dS K_j                                      (A = dS K-major, B = K_j MN-major) -> TMEM dQ
//   softmax warps: dQ tile -> shared memory -> TMA reduce-add (fp32, done by the L2) into dQacc[b, i*128.., h*64..];
//               a 3-D tensor map [B][N][D] clips the rows beyond the image.
// The same shared-memory image of P / dS serves as MN-major A (dV, dK) and as K-major A (dQ): no transposes.
// dK_j, dV_j leave through registers as 16-bit values into the dQKV activation; dQacc is converted by dq_convert_kernel.
// Head_dim 128 (DH = 128): every item also names one 64-column half of the head, and dK / dV / dQ of that half are its only
// outputs, so the TMEM map above (S 128 | dP 128 | dV 64 | dK 64 | dQ 64) and the drains stay as they are; S and dP contract over
// all 128 columns (8 k-steps across the two swizzle atoms of every tile).  The two halves of a key block recompute the same
// P / dS: twice the exponentials of one pass, against a 128-column dQ that has no room in TMEM next to 128-key S, dP, dV and dK.
// A [128 x 128] tile is 32 KB, so K / V and Q / dO get one shared-memory slot each (211 KB in all) and the MMA warp issues the
// next tile's S / dP only after the current tile's dV / dK / dQ (AbwCfg::ONE_SLOT): its operands land in the slot those free.
// F16 = true: fp16 Q / K / V / dO operands (fp16 engines); P and dS are packed to fp16 with satfinite, dK / dV leave as fp16.
// Warp roles: warps 0..7 softmax/drain (quadrant = warp % 4, key-column half = warp / 4: two warps per scheduler hide each
// other's MUFU / TMEM latencies -- the backward needs no row reductions, so a row splits freely), warp 8 = TMA producer,
// warp 9 = MMA issuer + TMEM allocator.  Ragged tails are trimmed: a short key block runs S / dP at N = 32 per 32 keys and
// only the dQ k-steps that hold keys; a short query tile only the dV / dK k-steps that hold queries.
#pragma once
#include "ptx.cuh"

namespace vitocm {

struct AttnBwdArgs {
  int n_tokens;       // N
  int embed_dim;      // D = H * DH
  int heads;
  float scale;        // qk scale
  float scale_log2;   // scale * log2(e)
  const float* lse2;  // [B][H][Npad], Npad = N rounded up to 128; +inf in the pad rows
  const float* delta; // [B][H][Npad]; 0 in the pad rows
  __nv_bfloat16* dqkv;  // [B*N][ld]: dK at column D + h*DH, dV at 2D + h*DH (dQ comes from dq_convert_kernel)
  long long ld;
  int n_items;        // work items = (DH / 64 column halves x) key blocks x heads x images; persistent CTAs walk them with stride gridDim.x
  int debug;          // diagnostics (VITOCM_ABW_DEBUG): 1 = skip the dQ reduce-add, 2 = timeline stamps
};

constexpr int ABW_SM_WARPS = 8;    // softmax / drain warps: two per TMEM lane quadrant, each takes half of the key columns
constexpr int ABW_DRAIN_WARP0 = 8;   // warps 8..11: dQ drain (one per TMEM lane quadrant)
constexpr int ABW_TMA_WARP = 12, ABW_MMA_WARP = 13;   // warps 14, 15 idle (setmaxnreg works on whole warpgroups)
constexpr int ABW_THREADS = 512;
constexpr int ABW_REGS_SOFTMAX = 200, ABW_REGS_OTHER = 56;   // 8 x 32 x 200 + 8 x 32 x 56 = 64 K registers
constexpr int ABW_TILE = 128 * 64 * 2;          // 16 KB: [128 rows][64 bf16]
constexpr int ABW_S_COL = 0, ABW_DP_COL = 128, ABW_DV_COL = 256, ABW_DK_COL = 320, ABW_DQ_COL = 384;
constexpr int ABW_TMEM_COLS = 512;
// shared memory: (K, V) x 2 | (Q, dO) x 2 | P (2 atoms) | dS (2 atoms) | dQ staging (4 warps x 4 KB) | row statistics | barriers
constexpr int ABW_STAT_BYTES = 2 * 1024;   // [2 slots][LSE2 | Delta][128 rows] fp32
constexpr int ABW_DQ_STG_BYTES = 4 * 4096;
constexpr int ABW_SMEM_BYTES = 4 * ABW_TILE + 4 * ABW_TILE + 2 * ABW_TILE + 2 * ABW_TILE + ABW_DQ_STG_BYTES + ABW_STAT_BYTES + 1024 + 256;

template <int DH>
struct AbwCfg {
  static_assert(DH == 64 || DH == 128, "head_dim 64 or 128");
  static constexpr int ATOMS = DH / 64;              // 64-column swizzle atoms per tile row; also column halves per item
  static constexpr int TILE = ATOMS * ABW_TILE;      // one [128 x DH] bf16 tile
  static constexpr int SLOTS = DH == 64 ? 2 : 1;     // K / V and Q / dO slots
  static constexpr bool ONE_SLOT = SLOTS == 1;
  static constexpr int SMEM_BYTES = SLOTS * 2 * TILE + SLOTS * 2 * TILE + 2 * ABW_TILE + 2 * ABW_TILE + ABW_DQ_STG_BYTES + ABW_STAT_BYTES + 1024 + 256;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
};
static_assert(AbwCfg<64>::SMEM_BYTES == ABW_SMEM_BYTES, "head_dim 64 layout");

// diagnostics (VITOCM_ABW_DEBUG=2): SM-clock stamps of CTA (1,0,0) -- [role 0 = softmax warp 0, 1 = MMA thread][query tile < 8][event < 8]
__device__ long long g_abw_timeline[2 * 8 * 8];
__device__ __forceinline__ void abw_stamp(bool on, int role, int i, int ev) {
  if (on && i < 8) g_abw_timeline[(role * 8 + i) * 8 + ev] = clock64();
}

__device__ __forceinline__ void tma_reduce_add_3d(const CUtensorMap* tmap, uint32_t smem_src, int c0, int c1, int c2) {
  asm volatile("cp.reduce.async.bulk.tensor.3d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}

template <int DH = 64, bool F16 = false>
__global__ void __launch_bounds__(ABW_THREADS, 1)
attn_bwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_do,
                        const __grid_constant__ CUtensorMap tmap_dq, const AttnBwdArgs args) {
  using Cfg = AbwCfg<DH>;
  constexpr int ATOMS = Cfg::ATOMS, TILE = Cfg::TILE, SLOTS = Cfg::SLOTS;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_kv = smem;                          // [SLOTS][K | V]
  const uint32_t smem_qdo = smem_kv + SLOTS * 2 * TILE;   // [SLOTS][Q | dO]
  const uint32_t smem_p = smem_qdo + SLOTS * 2 * TILE;    // [2 atoms of 64 keys][128 q][128 B]
  const uint32_t smem_ds = smem_p + 2 * ABW_TILE;
  const uint32_t smem_dq = smem_ds + 2 * ABW_TILE;        // fp32 staging, one 32 x 32 box per drain warp
  const uint32_t smem_stat = smem_dq + ABW_DQ_STG_BYTES;  // per query tile: LSE2 and Delta rows (bulk-copied by the producer)
  const uint32_t bars = smem_stat + ABW_STAT_BYTES;
  const uint32_t kv_full = bars;            // [2] K_j, V_j of an item landed
  const uint32_t kv_empty = bars + 16;      // [2] all MMAs reading that K / V slot retired
  const uint32_t qdo_full = bars + 32;      // [2]
  const uint32_t qdo_empty = bars + 48;     // [2]
  const uint32_t sdp_full = bars + 64;      // MMA -> softmax: S, dP complete
  const uint32_t pds_full = bars + 72;      // softmax -> MMA: P, dS in shared memory (ABW_SM_WARPS arrivals)
  const uint32_t dq_full = bars + 80;       // MMA -> softmax / drain: dQ of a tile complete (also: P / dS / dV / dK MMAs retired)
  const uint32_t dq_empty = bars + 88;      // drain -> MMA: dQ columns drained (4 warps)
  const uint32_t sdp_free = bars + 96;      // softmax -> MMA: S, dP columns are in registers (ABW_SM_WARPS arrivals)
  const uint32_t dkv_empty = bars + 104;    // softmax -> MMA: dK / dV of the finished item are in registers (ABW_SM_WARPS arrivals)
  const uint32_t tmem_ptr_smem = bars + 112;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int N = args.n_tokens, D = args.embed_dim;
  const int n_q = (N + 127) / 128;           // query tiles per item == key blocks per (image, head)
  // this CTA's items: blockIdx.x, blockIdx.x + gridDim.x, ...; tiles are numbered t = w * n_q + i across them
  const int my_items = (args.n_items - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int T = my_items * n_q;
  auto item_of = [&](int w, int& j, int& h, int& b, int& hc) {   // hc: first column of the item's half inside the head
    int it = blockIdx.x + w * gridDim.x;
    hc = 0;
    if (ATOMS == 2) {
      hc = (it & 1) * 64;
      it >>= 1;
    }
    j = it % n_q;
    h = (it / n_q) % args.heads;
    b = it / (n_q * args.heads);
  };
  auto kv_len_of = [&](int j) {
    const int len = N - j * 128;
    return len > 128 ? 128 : len;
  };

  if (warp == ABW_TMA_WARP && lane == 0) {
    ptx::prefetch_tmap(&tmap_qkv);
    ptx::prefetch_tmap(&tmap_do);
    ptx::prefetch_tmap(&tmap_dq);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(kv_full + 8 * s, 1);
      ptx::mbar_init(kv_empty + 8 * s, 1);
      ptx::mbar_init(qdo_full + 8 * s, 1);
      ptx::mbar_init(qdo_empty + 8 * s, 1);
    }
    ptx::mbar_init(sdp_full, 1);
    ptx::mbar_init(sdp_free, ABW_SM_WARPS);
    ptx::mbar_init(pds_full, ABW_SM_WARPS);
    ptx::mbar_init(dq_full, 1);
    ptx::mbar_init(dq_empty, 4);
    ptx::mbar_init(dkv_empty, ABW_SM_WARPS);
    ptx::fence_barrier_init();
  }
  if (warp == ABW_MMA_WARP) {
    ptx::tmem_alloc(tmem_ptr_smem, ABW_TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::lds_u32(tmem_ptr_smem);

  if (warp >= ABW_SM_WARPS) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(ABW_REGS_OTHER));
  if (warp == ABW_TMA_WARP) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      for (int w = 0; w < my_items; ++w) {
        int j, h, b, hc;
        item_of(w, j, h, b, hc);
        const int row_base = b * N;
        const int ks = w & (SLOTS - 1);
        ptx::mbar_wait(kv_empty + 8 * ks, ((w >> (SLOTS - 1)) & 1) ^ 1, 40);
        ptx::mbar_arrive_expect_tx(kv_full + 8 * ks, 2 * TILE);
        for (int at = 0; at < ATOMS; ++at) {
          ptx::tma_load_2d(smem_kv + ks * 2 * TILE + at * ABW_TILE, &tmap_qkv, kv_full + 8 * ks, D + h * DH + at * 64, row_base + j * 128);
          ptx::tma_load_2d(smem_kv + ks * 2 * TILE + TILE + at * ABW_TILE, &tmap_qkv, kv_full + 8 * ks, 2 * D + h * DH + at * 64,
                           row_base + j * 128);
        }
        const long long stat_base = (static_cast<long long>(b) * args.heads + h) * (n_q * 128);
        for (int i = 0; i < n_q; ++i) {
          const int t = w * n_q + i, slot = t & (SLOTS - 1);
          ptx::mbar_wait(qdo_empty + 8 * slot, ((t >> (SLOTS - 1)) & 1) ^ 1, 41);
          ptx::mbar_arrive_expect_tx(qdo_full + 8 * slot, 2 * TILE + 1024);
          ptx::bulk_load_1d(smem_stat + slot * 1024, args.lse2 + stat_base + i * 128, 512, qdo_full + 8 * slot);
          ptx::bulk_load_1d(smem_stat + slot * 1024 + 512, args.delta + stat_base + i * 128, 512, qdo_full + 8 * slot);
          for (int at = 0; at < ATOMS; ++at) {
            ptx::tma_load_2d(smem_qdo + slot * 2 * TILE + at * ABW_TILE, &tmap_qkv, qdo_full + 8 * slot, h * DH + at * 64, row_base + i * 128);
            ptx::tma_load_2d(smem_qdo + slot * 2 * TILE + TILE + at * ABW_TILE, &tmap_do, qdo_full + 8 * slot, h * DH + at * 64,
                             row_base + i * 128);
          }
        }
      }
    }
  } else if (warp == ABW_MMA_WARP) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      constexpr uint32_t FMT = F16 ? 0u : 1u;
      constexpr uint32_t idesc_t = ptx::make_idesc(128, 64, true, true, FMT);      // dV, dK: A (P / dS) and B (dO / Q) MN-major
      constexpr uint32_t idesc_q = ptx::make_idesc(128, 64, false, true, FMT);     // dQ: A = dS K-major, B = K_j MN-major
      const uint64_t p_desc_mn = ptx::make_smem_desc_sw128(smem_p, 1024, ABW_TILE);    // 64-key atoms 16 KB apart
      const uint64_t ds_desc_mn = ptx::make_smem_desc_sw128(smem_ds, 1024, ABW_TILE);
      const uint64_t ds_desc_k = ptx::make_smem_desc_sw128(smem_ds, 1024, 0);
      // S = Q K^T and dP = dO V^T of tile t (item w = t / n_q); only the 32-key chunks that hold keys
      auto issue_sdp = [&](int t) {
        const int w = t / n_q, i = t - w * n_q, slot = t & (SLOTS - 1), ks = w & (SLOTS - 1);
        int j, h, b, hc;
        item_of(w, j, h, b, hc);
        if (i == 0) ptx::mbar_wait(kv_full + 8 * ks, (w >> (SLOTS - 1)) & 1, 42);
        ptx::mbar_wait(qdo_full + 8 * slot, (t >> (SLOTS - 1)) & 1, 41);
        ptx::tc_fence_after();
        const uint32_t idesc_s = ptx::make_idesc(128, ((kv_len_of(j) + 31) >> 5) * 32, false, false, FMT);
        const uint64_t k_desc = ptx::make_smem_desc_sw128(smem_kv + ks * 2 * TILE, 1024, 0);
        const uint64_t v_desc = ptx::desc_advance(k_desc, TILE);
        const uint64_t q_desc = ptx::make_smem_desc_sw128(smem_qdo + slot * 2 * TILE, 1024, 0);
        const uint64_t do_desc = ptx::desc_advance(q_desc, TILE);
        // k step = 16 columns: 32 B inside a swizzle atom, the next atom every 4 steps
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          ptx::umma_bf16_ss(tmem_base + ABW_S_COL, ptx::desc_advance(q_desc, (k >> 2) * ABW_TILE + (k & 3) * 32),
                            ptx::desc_advance(k_desc, (k >> 2) * ABW_TILE + (k & 3) * 32), idesc_s, k ? 1u : 0u);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k)
          ptx::umma_bf16_ss(tmem_base + ABW_DP_COL, ptx::desc_advance(do_desc, (k >> 2) * ABW_TILE + (k & 3) * 32),
                            ptx::desc_advance(v_desc, (k >> 2) * ABW_TILE + (k & 3) * 32), idesc_s, k ? 1u : 0u);
        ptx::umma_commit(sdp_full);
      };
      if (T > 0) issue_sdp(0);
      for (int t = 0; t < T; ++t) {
        const int w = t / n_q, i = t - w * n_q, slot = t & (SLOTS - 1), ks = w & (SLOTS - 1);
        int j, h, b, hc;
        item_of(w, j, h, b, hc);
        const int kv_len = kv_len_of(j);
        const bool tl = args.debug == 2 && blockIdx.x == 1 && w == 0;
        abw_stamp(tl, 1, i, 0);
        // the next tile's logits go first, as soon as the softmax warps hold S / dP of this tile in registers: they are ready
        // long before those warps finish tile t, and the tensor core runs dV / dK / dQ of tile t under the exponentials of t + 1
        // (one slot: the next tile's operands replace this tile's, so its S / dP follow this tile's MMAs below)
        if (!Cfg::ONE_SLOT && t + 1 < T) {
          ptx::mbar_wait(sdp_free, t & 1, 49);
          ptx::tc_fence_after();
          issue_sdp(t + 1);
        }
        ptx::mbar_wait(pds_full, t & 1, 43);     // P, dS of tile t in shared memory
        ptx::tc_fence_after();
        abw_stamp(tl, 1, i, 1);
        if (i == 0 && w > 0) {                   // dK / dV still hold the previous item until the softmax warps have read them out
          ptx::mbar_wait(dkv_empty, (w - 1) & 1, 51);
          ptx::tc_fence_after();
        }
        // MN-major B operands: the item's 64-column half (atom hc / 64) of Q_i, dO_i, K_j
        const uint64_t q_desc_mn = ptx::make_smem_desc_sw128(smem_qdo + slot * 2 * TILE + (hc / 64) * ABW_TILE, 1024, 1024);
        const uint64_t do_desc_mn = ptx::desc_advance(q_desc_mn, TILE);
        const uint64_t k_desc_mn = ptx::make_smem_desc_sw128(smem_kv + ks * 2 * TILE + (hc / 64) * ABW_TILE, 1024, 1024);
        const uint32_t acc0 = i > 0 ? 1u : 0u;
        int q_len = N - i * 128;
        q_len = q_len > 128 ? 128 : q_len;
        const int qsteps = (q_len + 15) >> 4;      // 16-row steps that hold queries (P = dS = 0 beyond q_len inside them)
        // dV += P^T dO_i,  dK += dS^T Q_i: 16 query rows (2048 B of every atom) per MMA
        if (qsteps == 8) {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            ptx::umma_bf16_ss(tmem_base + ABW_DV_COL, ptx::desc_advance(p_desc_mn, k * 2048), ptx::desc_advance(do_desc_mn, k * 2048), idesc_t, k ? 1u : acc0);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            ptx::umma_bf16_ss(tmem_base + ABW_DK_COL, ptx::desc_advance(ds_desc_mn, k * 2048), ptx::desc_advance(q_desc_mn, k * 2048), idesc_t, k ? 1u : acc0);
        } else {
#pragma unroll 1
          for (int k = 0; k < qsteps; ++k)
            ptx::umma_bf16_ss(tmem_base + ABW_DV_COL, ptx::desc_advance(p_desc_mn, k * 2048), ptx::desc_advance(do_desc_mn, k * 2048), idesc_t, k ? 1u : acc0);
#pragma unroll 1
          for (int k = 0; k < qsteps; ++k)
            ptx::umma_bf16_ss(tmem_base + ABW_DK_COL, ptx::desc_advance(ds_desc_mn, k * 2048), ptx::desc_advance(q_desc_mn, k * 2048), idesc_t, k ? 1u : acc0);
        }
        ptx::umma_commit(qdo_empty + 8 * slot);   // Q_i / dO_i no longer needed
        // dQ_i = dS K_j: 16 keys per MMA (32 B inside a 64-key atom of dS; 2048 B of K_j)
        if (t > 0) {
          ptx::mbar_wait(dq_empty, (t - 1) & 1, 44);
          ptx::tc_fence_after();
        }
        if (kv_len == 128) {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            ptx::umma_bf16_ss(tmem_base + ABW_DQ_COL, ptx::desc_advance(ds_desc_k, (k >> 2) * ABW_TILE + (k & 3) * 32),
                              ptx::desc_advance(k_desc_mn, k * 2048), idesc_q, k ? 1u : 0u);
        } else {
          const int ksteps = (kv_len + 15) >> 4;   // dS = 0 beyond kv_len inside the last step
#pragma unroll 1
          for (int k = 0; k < ksteps; ++k)
            ptx::umma_bf16_ss(tmem_base + ABW_DQ_COL, ptx::desc_advance(ds_desc_k, (k >> 2) * ABW_TILE + (k & 3) * 32),
                              ptx::desc_advance(k_desc_mn, k * 2048), idesc_q, k ? 1u : 0u);
        }
        ptx::umma_commit(dq_full);
        if (i == n_q - 1) ptx::umma_commit(kv_empty + 8 * ks);   // last reader of this K / V slot
        abw_stamp(tl, 1, i, 2);
        if (Cfg::ONE_SLOT && t + 1 < T) {
          ptx::mbar_wait(sdp_free, t & 1, 49);
          ptx::tc_fence_after();
          issue_sdp(t + 1);
        }
      }
    }
  } else if (warp >= ABW_DRAIN_WARP0 && warp < ABW_DRAIN_WARP0 + 4) {
    // ===================== dQ drain warps =====================
    // dQ of tile t: TMEM -> fp32 box -> reduce-add into dQacc[b, i*128 + q*32 .., h*64 ..]; off the softmax warps' path
    const int q = warp & 3;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t stg = smem_dq + q * 4096;
    const int sw = lane & 7;
    for (int t = 0; t < T; ++t) {
      const int w = t / n_q, i = t - w * n_q;
      int j, h, b, hc;
      item_of(w, j, h, b, hc);
      ptx::mbar_wait(dq_full, t & 1, 46);
      ptx::tc_fence_after();
      const bool store = i * 128 + q * 32 < N && args.debug != 1;
#pragma unroll
      for (int hb = 0; hb < 2; ++hb) {           // one 32-column box at a time through one staging box
        uint32_t t0[32];
        ptx::tmem_ld_32x32b_x32(lane_addr + ABW_DQ_COL + hb * 32, t0);
        ptx::tmem_ld_wait(t0);
        if (hb == 1) {                           // both halves are out of TMEM: dQ columns free (before any wait on the box)
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(dq_empty);
        }
        if (lane == 0) ptx::bulk_wait_read0();   // the previous reduce has finished reading the box
        __syncwarp();
#pragma unroll
        for (int g = 0; g < 8; ++g) ptx::sts_v4(stg + lane * 128 + ((g ^ sw) << 4), t0[4 * g], t0[4 * g + 1], t0[4 * g + 2], t0[4 * g + 3]);
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && store) {
          tma_reduce_add_3d(&tmap_dq, stg, h * DH + hc + hb * 32, i * 128 + q * 32, b);
          ptx::bulk_commit();
        }
      }
    }
    if (lane == 0) ptx::bulk_wait_all0();
  } else if (warp < ABW_SM_WARPS) {
    // ===================== softmax warps (0 .. ABW_SM_WARPS-1) =====================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(ABW_REGS_SOFTMAX));
    const int q = warp & 3;
    const int half = warp >> 2;    // which half of the key columns (S / dP phase), and dK (0) or dV (1) at the end of an item
    const int r = q * 32 + lane;   // query row inside the tile (S, dP phases) or key row (dK / dV drain)
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float sl2 = args.scale_log2;
    const uint64_t sl2_2 = ptx::dup_f32x2(sl2);
    const uint64_t sc_2 = ptx::dup_f32x2(args.scale);
    // dK_j (warps 0..3) / dV_j (warps 4..7) of item w: TMEM -> registers -> bf16 rows of dQKV.  Called once all MMAs of the item
    // have retired (dq_full of its last tile); the MMA warp may overwrite the accumulators after the dkv_empty arrive.
    auto drain_dkv = [&](int w) {
      int j, h, b, hc;
      item_of(w, j, h, b, hc);
      const int kv_len = kv_len_of(j);
      __nv_bfloat16* o = args.dqkv + static_cast<long long>(b * N + j * 128 + r) * args.ld + h * DH + hc + (half == 0 ? D : 2 * D);
      uint32_t t0[32], t1[32];
      ptx::tmem_ld_32x32b_x32(lane_addr + (half == 0 ? ABW_DK_COL : ABW_DV_COL), t0);        // warp-collective
      ptx::tmem_ld_32x32b_x32(lane_addr + (half == 0 ? ABW_DK_COL : ABW_DV_COL) + 32, t1);
      ptx::tmem_ld_wait(t0);
      ptx::tmem_ld_wait(t1);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(dkv_empty);
      if (r < kv_len) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          reinterpret_cast<uint4*>(o)[g] =
              make_uint4(ptx::pack_h2<F16>(__uint_as_float(t0[8 * g]), __uint_as_float(t0[8 * g + 1])),
                         ptx::pack_h2<F16>(__uint_as_float(t0[8 * g + 2]), __uint_as_float(t0[8 * g + 3])),
                         ptx::pack_h2<F16>(__uint_as_float(t0[8 * g + 4]), __uint_as_float(t0[8 * g + 5])),
                         ptx::pack_h2<F16>(__uint_as_float(t0[8 * g + 6]), __uint_as_float(t0[8 * g + 7])));
          reinterpret_cast<uint4*>(o + 32)[g] =
              make_uint4(ptx::pack_h2<F16>(__uint_as_float(t1[8 * g]), __uint_as_float(t1[8 * g + 1])),
                         ptx::pack_h2<F16>(__uint_as_float(t1[8 * g + 2]), __uint_as_float(t1[8 * g + 3])),
                         ptx::pack_h2<F16>(__uint_as_float(t1[8 * g + 4]), __uint_as_float(t1[8 * g + 5])),
                         ptx::pack_h2<F16>(__uint_as_float(t1[8 * g + 6]), __uint_as_float(t1[8 * g + 7])));
        }
      }
    };
    for (int t = 0; t < T; ++t) {
      const int w = t / n_q, i = t - w * n_q;
      int j, h, b, hc;
      item_of(w, j, h, b, hc);
      const int kv_len = kv_len_of(j);
      const int nch = (kv_len + 31) >> 5;          // 32-key chunks of this key block that hold keys
      const bool tl = args.debug == 2 && blockIdx.x == 1 && w == 0 && lane == 0;
      abw_stamp(tl && warp == 0, 0, i, 6);
      // row statistics of this query tile from shared memory (rows beyond the image: LSE2 = +inf -> P = 0 -> dS = 0; dP is
      // finite there: the rows hold other tokens or zeros)
      ptx::mbar_wait(qdo_full + 8 * (t & (SLOTS - 1)), (t >> (SLOTS - 1)) & 1, 50);
      const float lse = ptx::lds_f32(smem_stat + (t & (SLOTS - 1)) * 1024 + r * 4);
      const float dlt = ptx::lds_f32(smem_stat + (t & (SLOTS - 1)) * 1024 + 512 + r * 4);
      const uint64_t nlse_2 = ptx::dup_f32x2(-lse);
      const uint64_t ndl_2 = ptx::dup_f32x2(-dlt * args.scale);
      abw_stamp(tl && warp == 0, 0, i, 0);
      ptx::mbar_wait(sdp_full, t & 1, 45);
      ptx::tc_fence_after();
      abw_stamp(tl && warp == 0, 0, i, 1);
      // ---- P = exp2(S * sl2 - LSE2), dS = P * (dP * scale - Delta * scale) for this warp's (up to) two 32-key chunks, on the
      //      packed f32x2 pipe; results wait in registers until the previous tile's MMAs have released the P / dS buffers
      uint32_t sv[2][32], dp[2][32];   // S / dP, then (in place, first 16 words of each) the packed bf16 P / dS
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c = 2 * half + cc;
        if (c < nch) {
          ptx::tmem_ld_32x32b_x32(lane_addr + ABW_S_COL + c * 32, sv[cc]);
          ptx::tmem_ld_32x32b_x32(lane_addr + ABW_DP_COL + c * 32, dp[cc]);
        }
      }
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        if (2 * half + cc < nch) {
          ptx::tmem_ld_wait(sv[cc]);
          ptx::tmem_ld_wait(dp[cc]);
        }
      }
      ptx::tc_fence_before();     // S / dP are in registers: the MMA warp may overwrite the columns with the next tile's
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(sdp_free);
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c = 2 * half + cc;
        if (c < nch) {
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            const uint64_t a2 = ptx::fma_f32x2(ptx::pack_f32x2(__uint_as_float(sv[cc][2 * u]), __uint_as_float(sv[cc][2 * u + 1])), sl2_2, nlse_2);
            float a0, a1;
            ptx::unpack_f32x2(a2, a0, a1);
            const float p0 = ptx::ex2_approx(a0), p1 = ptx::ex2_approx(a1);
            const uint64_t g2 = ptx::fma_f32x2(ptx::pack_f32x2(__uint_as_float(dp[cc][2 * u]), __uint_as_float(dp[cc][2 * u + 1])), sc_2, ndl_2);
            const uint64_t d2 = ptx::mul_f32x2(ptx::pack_f32x2(p0, p1), g2);
            float d0, d1;
            ptx::unpack_f32x2(d2, d0, d1);
            sv[cc][u] = ptx::pack_h2<F16>(p0, p1);     // words u <= 2u have been consumed
            dp[cc][u] = ptx::pack_h2<F16>(d0, d1);
          }
          if (c * 32 + 32 > kv_len) {   // ragged key block: keys beyond the image contribute nothing
#pragma unroll
            for (int u = 0; u < 16; ++u) {
              const int k0 = c * 32 + 2 * u;
              const uint32_t keep = (k0 < kv_len ? 0x0000ffffu : 0u) | (k0 + 1 < kv_len ? 0xffff0000u : 0u);
              sv[cc][u] &= keep;
              dp[cc][u] &= keep;
            }
          }
        }
      }
      abw_stamp(tl && warp == 0, 0, i, 2);
      if (t > 0) {   // previous tile's dV / dK / dQ MMAs retired: P / dS may be overwritten
        ptx::mbar_wait(dq_full, (t - 1) & 1, 47);
        if (i == 0) {   // ... and it closed an item: its dK / dV leave now, under the tensor core's work on this item
          ptx::tc_fence_after();
          drain_dkv(w - 1);
        }
      }
      abw_stamp(tl && warp == 0, 0, i, 3);
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        const int c = 2 * half + cc;
        if (c < nch) {
          // 32 keys = 4 chunks of 16 B in row r of atom c / 2 (SWIZZLE_128B: chunk ^ (r & 7))
          const uint32_t off = (c >> 1) * ABW_TILE + r * 128;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const uint32_t ch = static_cast<uint32_t>((((c & 1) * 4 + g) ^ (r & 7)) << 4);
            ptx::sts_v4(smem_p + off + ch, sv[cc][4 * g], sv[cc][4 * g + 1], sv[cc][4 * g + 2], sv[cc][4 * g + 3]);
            ptx::sts_v4(smem_ds + off + ch, dp[cc][4 * g], dp[cc][4 * g + 1], dp[cc][4 * g + 2], dp[cc][4 * g + 3]);
          }
        }
      }
      ptx::fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(pds_full);
      abw_stamp(tl && warp == 0, 0, i, 4);
    }
    if (T > 0) {
      ptx::mbar_wait(dq_full, (T - 1) & 1, 48);
      ptx::tc_fence_after();
      drain_dkv(my_items - 1);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == ABW_MMA_WARP) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, ABW_TMEM_COLS);
  }
}

}  // namespace vitocm
