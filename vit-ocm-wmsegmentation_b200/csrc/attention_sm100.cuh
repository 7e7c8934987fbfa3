// Flash-style multi-head self-attention for sm_100a (head_dim DH = 64 or 128), tcgen05 + TMEM + TMA:
//     ctx[b, i, h*DH:(h+1)*DH] = softmax_j( scale * q_i . k_j ) @ v        (never materialises N x N)
// Replaces SSS/dino/vision_transformer.py:83-87 (q@k^T*scale, softmax, attn@v, transpose/reshape)
// for the blocks whose attention matrix is not returned.
//
// One work item = one (image b, head h, 128-query tile); CTAs are persistent and walk the items.  q/k/v are read straight out of the fused
// QKV activation [B*N, ld] (bf16, columns [3][H][DH]) by one 2-D TMA tensor map (box 64 x 128,
// SWIZZLE_128B; DH / 64 boxes per tile).  Warp roles (256 threads): warps 0..3 = softmax (one thread per query row; TMEM lane
// quadrant = warp % 4), warp 4 = TMA producer, warp 5 = MMA issuer + TMEM allocator, warps 6..7 idle.
// setmaxnreg moves registers from warpgroup 1 to the softmax warpgroup (208 vs 48 per thread in bf16 mode).
//   S = Q K_j^T      : tcgen05.mma  M128 x N(<=128) x K(DH), both operands K-major, into TMEM
//   softmax          : one tcgen05.ld pass of S into registers; scale/shift on the packed f32x2 pipe
//                      (FFMA2), MUFU.EX2, row sums on FADD2, P -> TMEM (tcgen05.st, packed bf16x2 columns):
//                      no shared-memory round trip, no generic->async proxy fence
//   O += P V_j       : tcgen05.mma  M128 x N(DH) x K(<=128), A = P from TMEM, B = V (smem, MN-major),
//                      accumulating in TMEM
// The running maximum is only raised when a row exceeds it by more than 2^8 ("lazy rescale"): softmax
// is shift invariant, so a stale maximum changes nothing but keeps O in TMEM untouched in the
// common case; when it is raised the softmax warps rescale their O rows in TMEM.
// At head_dim 64 two CTAs are co-resident per SM (65 KB smem, 256 TMEM columns each: S 128 | O 64 | P 64) so one CTA's MMAs
// overlap the other's exponentials; head_dim 128 runs one CTA per SM (AttnCfg, DESIGN.md section 3).
// Ragged query tail ("packed" items): N = 785 leaves 17 query rows per (image, head) beyond the last full tile; a tile of
// its own would spend a full tile's exponentials on them (1/7 of the kernel).  Instead the tails of `pack` = 4 (<= 32 rows)
// or 2 (<= 64 rows) consecutive (image, head) pairs share ONE 128-row tile, one 32- or 64-lane slot each: the S and PV MMAs
// are issued once per slot against that pair's own K / V with a disable-output-lane mask that leaves the other slots'
// TMEM lanes untouched, and the softmax warps run unchanged (one thread per row, whichever pair the row belongs to).
// The slot logic only exists in the PACKED = true instantiations; launches without packed items (no ragged tail, a tail
// of more than 64 rows, or more than 16 full tiles per pair) run PACKED = false, where every item is an ordinary tile.
// SPLIT = true is the fp32-parity mode: every operand is a bf16 (hi, lo) pair and each product is
// hi*hi + hi*lo + lo*hi (fp32 accumulate in TMEM).
#pragma once
#include <type_traits>

#include "ptx.cuh"

namespace vitocm {

struct AttnArgs {
  int n_items;       // work items (persistent CTAs walk them with stride gridDim.x): groups of `pack` (image, head) pairs,
                     // each group = pack x n_fullq full query tiles (tile fastest) + one tail item when N % 128 != 0
  int n_qtiles, heads;   // n_qtiles = ceil(N / 128): rows per (image, head) of lse2 = n_qtiles * 128
  int n_fullq;       // full 128-row query tiles per pair = N / 128
  int pack;          // pairs sharing a tail item: 1 (the tail is an ordinary tile, or there is none), 2 or 4
  int group_items;   // pack * n_fullq + (N % 128 != 0)
  int n_pairs;       // images x heads
  int n_tokens;      // N per image (785 for 224^2 / patch 8)
  int embed_dim;     // D = H * head_dim
  int lo_col_off;    // SPLIT: column offset of the lo halves inside the qkv activation (= 3D)
  float scale_log2;  // qk scale * log2(e)
  __nv_bfloat16* out;  // ctx [B*N, ldo]
  long long ldo;
  int out_lo_off;    // SPLIT: column offset of the lo half of ctx
  float* lse2;       // training: [B][H][Npad] (Npad = N rounded up to 128) log2-sum-exp of the scaled logits
                     // (max * scale_log2 + log2 l); +inf in the pad rows; or nullptr
  int track_max;        // 1 = round-1 behaviour: every KV block's row maximum is computed (128 FMNMX per thread and block) to detect a
                        // row rising above the maximum in use; 0 (default) = only block 0's maximum is computed; later blocks
                        // are checked through their row SUM of exponentials (one compare + vote): while no sum exceeds
                        // 2^ATT_SUM_TRIGGER no single exponential can have overflowed the 16-bit P format, and a stale maximum is
                        // exact otherwise (softmax is shift invariant, O and l accumulate in fp32).  Only a block that trips
                        // the trigger pays for row_max(), the rescale of O and a second pass of exponentials.
  int n_full_items;     // attn_fwd_quad_kernel: items [0, n_full_items) are full query tiles, items beyond it the packed tails of `pack` pairs each
  int ctrl_hoist;       // attn_fwd_quad_kernel: 1 = PV_j / S_{j+1} operands prepared before the wait for P_j (VITOCM_ATTN_HOIST, A/B knob)
  int tails_only;       // 1 = the launch covers only the ragged query tail of every pair (item i = the tail item of group i); the full
                        // tiles are computed by attn_fwd_quad_kernel (attention_quad_sm100.cuh)
  int timeline_item;    // diagnostics: which of a CTA's work items (0, 1, ...) the stamps are taken on
  long long* timeline;  // diagnostics (vitocm_attention_timeline) or nullptr: clock64 stamps of CTAs (0,0,0) and (1,0,0)
  int stagger_clk;      // attn_fwd_quad_kernel: CTA k starts k / gridDim.x x stagger_clk SM clocks late (VITOCM_ATTN_STAGGER) -- every CTA
                        // does the same work in the same time, so without it all of them load K / V and drain O in the same instants
};

// timeline layout: [cta 0..1][role 0 = softmax warp 0, 1 = MMA thread][kv block j < 16][event < 8]
constexpr int ATT_TL_EVENTS = 8;
constexpr int ATT_TL_BLOCKS = 16;
__device__ __forceinline__ void att_stamp(const AttnArgs& args, bool on, int role, int j, int ev, int pipe = -1) {
  if (pipe < 0) pipe = blockIdx.x;
  if (on && j < ATT_TL_BLOCKS) args.timeline[((pipe * 2 + role) * ATT_TL_BLOCKS + j) * ATT_TL_EVENTS + ev] = clock64();
}

constexpr int ATT_BQ = 128;
constexpr int ATT_BKV = 128;
constexpr int ATT_DH = 64;
constexpr int ATT_THREADS = 256;   // warpgroup 0 = softmax (warps 0..3), warpgroup 1 = TMA (warp 4) + MMA (warp 5)
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // 16 KB: one [128 x 64] bf16 tile
#ifndef VITOCM_ATT_RING
#define VITOCM_ATT_RING 3
#endif
constexpr int ATT_RING = VITOCM_ATT_RING;     // K / V tiles in flight (measured: 4 / 5 slots are 1-2 % slower, with or without packed tail items)
constexpr int ATT_S_COL = 0;      // S: 128 columns (fp32)
constexpr int ATT_O_COL = 128;    // O: 64 columns (fp32) at head_dim 64 (AttnCfg::O_COL / P_COL for either width)
constexpr int ATT_P_COL = 192;    // P: 64 columns of packed bf16x2 (128 keys); split mode: lo part in the next 64
constexpr float ATT_RESCALE_THRESHOLD = 8.0f;  // log2 units: raise the running maximum (rescale O, l) before the next block
constexpr float ATT_REDO_THRESHOLD = 60.0f;    // log2 units: exp2 of the current block may overflow -> redo it now
constexpr float ATT_REDO_THRESHOLD_F16 = 14.0f;   // fp16 P: 2^14 < 65504
// track_max == 0: a block whose row sum of exponentials exceeds this is redone against its true maximum.  bf16 P shares fp32's
// exponent range (trigger far below fp32 overflow of the sum and of O: 2^100 x 12 545 keys << 2^127); fp16 P must stay < 65504.
constexpr float ATT_SUM_TRIGGER = 1.2676506e30f;      // 2^100
constexpr float ATT_SUM_TRIGGER_F16 = 16384.0f;       // 2^14
constexpr int ATT_POLY_DEFAULT = 0;            // see run_attention (0: all MUFU, 1: 4/16 polynomial, 2: 7/16)

// DH = head_dim, 64 or 128.  A head row of 128 is two 128-byte swizzle atoms: every Q / K / V tile is ATOMS boxes of
// [128 rows x 64 columns], 16 KB apart; one part (hi or lo) of a tile = ATOMS x 16 KB.
// DH = 128 runs one CTA per SM: O takes 128 TMEM columns (S 128 | O 128 | P 64 [| P lo 64] <= 512), and Q + a 3-slot ring of
// 32 KB K / V blocks (2 slots of 64 KB in split mode) leaves no room for a second CTA's shared memory.
template <bool SPLIT, int DH = 64>
struct AttnCfg {
  static_assert(DH == 64 || DH == 128, "head_dim 64 or 128");
  static constexpr int ATOMS = DH / 64;
  static constexpr int NPART = SPLIT ? 2 : 1;                     // hi (+ lo)
  static constexpr int PART_BYTES = ATT_TILE_BYTES * ATOMS;       // one [128 x DH] bf16 tile
  static constexpr int SLOT_BYTES = PART_BYTES * NPART;           // one K or V block
  static constexpr int Q_BYTES = PART_BYTES * NPART;
  static constexpr int RING = (DH == 128 && SPLIT) ? 2 : ATT_RING;
  static constexpr int SMEM_BYTES = Q_BYTES + RING * SLOT_BYTES + 1024 + 256;   // + alignment slack + barrier block
  static constexpr bool ONE_CTA = SPLIT || DH == 128;             // one CTA per SM
  static constexpr int TMEM_COLS = ONE_CTA ? 512 : 256;
  static constexpr int O_COL = ATT_O_COL;                         // O: DH columns (fp32)
  static constexpr int P_COL = ATT_O_COL + DH;                    // P: 64 columns of packed bf16x2; split mode: lo part in the next 64
  // setmaxnreg budgets: 2 CTAs/SM x 128 x (208 + 48) = 64 K registers (bf16 at head_dim 64); one CTA/SM otherwise
  static constexpr int REGS_SOFTMAX = ONE_CTA ? 240 : 208;
  static constexpr int REGS_OTHER = ONE_CTA ? 64 : 48;
};

// work item -> (query tile, first pair, packed?); false = the item does not exist (pair beyond the batch in the last group)
template <bool PACKED>
__device__ __forceinline__ bool att_decode(const AttnArgs& a, int it, int& qt, int& pair0, bool& packed) {
  if (a.tails_only) {   // item = the tail of group `it` (one pair, or `pack` pairs sharing a tile)
    pair0 = it * a.pack;
    qt = a.n_fullq;
    packed = PACKED && a.pack > 1;
    return pair0 < a.n_pairs;
  }
  if (!PACKED) {   // launches without packed items (pack == 1): query tile fastest, then the pair; every item exists
    pair0 = it / a.n_qtiles;
    qt = it - pair0 * a.n_qtiles;
    packed = false;
    return true;
  }
  const int grp = it / a.group_items, r = it - grp * a.group_items;
  if (r < a.pack * a.n_fullq) {
    const int pi = r / a.n_fullq;
    pair0 = grp * a.pack + pi;
    qt = r - pi * a.n_fullq;
    packed = false;
  } else {
    pair0 = grp * a.pack;
    qt = a.n_fullq;
    packed = a.pack > 1;
  }
  return pair0 < a.n_pairs;
}
// disable-output-lane mask that leaves only slot s of nslots (2 or 4) equal lane groups writable
__device__ __forceinline__ void att_slot_mask(int s, int nslots, uint32_t (&m)[4]) {
#pragma unroll
  for (int w = 0; w < 4; ++w) m[w] = ((nslots == 4 ? w : (w >> 1)) == s) ? 0u : 0xffffffffu;   // set bit = lane not written
}

// POLY_MASK: bit i set = pair i of every 16 pairs of a 32-key chunk takes the FMA-pipe exp2 polynomial
// PACKED: the launch contains packed tail items (args.pack > 1); false compiles the slot logic out (every item is an ordinary tile)
// F16: q / k / v, P and ctx are IEEE fp16 instead of bf16 (fp16 engines): 11 significand bits at the same tensor-core rate.  P is
//      exp2 of (logit - running maximum) <= 2^ATT_RESCALE_THRESHOLD, or <= 2^redo threshold inside one block: the redo threshold
//      drops to 14 so that P stays below fp16's 65504; below 6e-8 P flushes to zero, like everything under 2^-24 of the row sum.
// DH: head_dim (64 or 128, see AttnCfg)
template <bool SPLIT, uint32_t POLY_MASK, bool PACKED, bool F16 = false, int DH = 64>
__global__ void __launch_bounds__(ATT_THREADS, AttnCfg<SPLIT, DH>::ONE_CTA ? 1 : 2)
attn_fwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_qkv, const __grid_constant__ CUtensorMap tmap_q32, const AttnArgs args) {
  using Cfg = AttnCfg<SPLIT, DH>;
  constexpr int NPART = Cfg::NPART;
  constexpr int ATOMS = Cfg::ATOMS;
  constexpr int RING = Cfg::RING;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t smem_q = smem;
  const uint32_t smem_ring = smem_q + Cfg::Q_BYTES;
  const uint32_t bars = smem_ring + RING * Cfg::SLOT_BYTES;
  const uint32_t q_full = bars;             // [1]
  const uint32_t kv_full = bars + 8;        // [RING]
  const uint32_t kv_empty = kv_full + 8 * RING;   // [RING]
  const uint32_t s_full = kv_empty + 8 * RING;    // MMA -> softmax
  const uint32_t s_empty = s_full + 8;      // softmax -> MMA   (4 warps)
  const uint32_t p_full = s_full + 16;      // softmax -> MMA   (4 warps)
  const uint32_t o_full = s_full + 24;      // MMA -> softmax
  const uint32_t q_empty = s_full + 32;     // MMA -> producer: all S MMAs of the work item retired (Q tile reusable)
  const uint32_t o_empty = s_full + 40;     // softmax -> MMA: O of the finished work item has been read (4 warps)
  const uint32_t tmem_ptr_smem = s_full + 48;
  static_assert(8 + 16 * RING + 56 <= 256, "barrier block overflows its 256 bytes");
  static_assert(Cfg::SMEM_BYTES <= 227 * 1024, "shared memory");

  // Persistent CTA: work items (query tile, head, image), query tile fastest so that the CTAs running side by side share
  // one image-head's K / V through L2.  Barriers, the K/V ring and TMEM live across items (all phase counters run on), so
  // the next item's Q / K loads and its first S MMA overlap the current item's last exponentials and its epilogue.
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int N = args.n_tokens;
  const int D = args.embed_dim;
  const int n_kv = (N + ATT_BKV - 1) / ATT_BKV;
  const bool tl0 = args.timeline != nullptr && blockIdx.x < 2 && (threadIdx.x & 31) == 0;

  if (warp == 4 && lane == 0) {
    ptx::prefetch_tmap(&tmap_qkv);
    ptx::prefetch_tmap(&tmap_q32);
    ptx::mbar_init(q_full, 1);
    for (int i = 0; i < RING; ++i) {
      ptx::mbar_init(kv_full + 8 * i, 1);
      ptx::mbar_init(kv_empty + 8 * i, 1);
    }
    ptx::mbar_init(s_full, 1);
    ptx::mbar_init(s_empty, 4);
    ptx::mbar_init(p_full, 4);
    ptx::mbar_init(o_full, 1);
    ptx::mbar_init(q_empty, 1);
    ptx::mbar_init(o_empty, 4);
    ptx::fence_barrier_init();
  }
  if (warp == 5) {
    ptx::tmem_alloc(tmem_ptr_smem, Cfg::TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::lds_u32(tmem_ptr_smem);
  if (tl0 && threadIdx.x == 0) args.timeline[((blockIdx.x * 2 + 0) * ATT_TL_BLOCKS + 15) * ATT_TL_EVENTS + 6] = clock64();   // CTA start

  if (warp >= 4) {
   asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(Cfg::REGS_OTHER));
   if (warp == 4) {
    // ===================== TMA producer =====================
    if (ptx::elect_one()) {
      int item = 0;   // K/V ring position, running across work items
      int w = 0;      // work items this CTA has processed
      for (int it = blockIdx.x; it < args.n_items; it += gridDim.x) {
      int qt, pair0;
      bool packed;
      if (!att_decode<PACKED>(args, it, qt, pair0, packed)) continue;
      const int nslots = (PACKED && packed) ? args.pack : 1;
      // pair of slot s (slots beyond the batch repeat the last pair: their rows are computed and dropped)
      auto pair_of = [&](int s) { const int pr = pair0 + s; return pr < args.n_pairs ? pr : args.n_pairs - 1; };
      ptx::mbar_wait(q_empty, (w & 1) ^ 1, 16);   // the previous item's S MMAs have retired
      ptx::mbar_arrive_expect_tx(q_full, Cfg::Q_BYTES);
      if (!PACKED || !packed) {
        const int b = pair0 / args.heads, h = pair0 - b * args.heads;
        for (int part = 0; part < NPART; ++part)
          for (int at = 0; at < ATOMS; ++at)
            ptx::tma_load_2d(smem_q + part * Cfg::PART_BYTES + at * ATT_TILE_BYTES, &tmap_qkv, q_full,
                             part * args.lo_col_off + h * DH + at * 64, b * N + qt * ATT_BQ);
      } else {
        // four 32-row boxes; slot s owns tile rows [s * 128 / nslots, (s + 1) * 128 / nslots) = the first rows of its pair's tail
        const int per = 4 / nslots;
        for (int part = 0; part < NPART; ++part)
          for (int at = 0; at < ATOMS; ++at)
            for (int u = 0; u < 4; ++u) {
              const int pr = pair_of(u / per);
              const int b = pr / args.heads, h = pr - b * args.heads;
              ptx::tma_load_2d(smem_q + part * Cfg::PART_BYTES + at * ATT_TILE_BYTES + u * 4096, &tmap_q32, q_full,
                               part * args.lo_col_off + h * DH + at * 64, b * N + qt * ATT_BQ + (u % per) * 32);
            }
      }
      // ring order = consumption order of the MMA warp: K0, K1, V0, K2, V1, ..., V_{n-1} (each entry = one tile per slot)
      int kv_col[4], kv_row[4];   // per slot: first column (head) and first row (image) of its pair's K / V, decoded once per item
      for (int sl = 0; sl < nslots; ++sl) {
        const int pr = pair_of(sl);
        const int b = pr / args.heads;
        kv_col[sl] = (pr - b * args.heads) * DH;
        kv_row[sl] = b * N;
      }
      auto load = [&](int which /*1 = K, 2 = V*/, int j) {
        for (int sl = 0; sl < nslots; ++sl) {
          const int slot = item % RING;
          const uint32_t parity = ((item / RING) & 1) ^ 1;
          ptx::mbar_wait(kv_empty + 8 * slot, parity, 10);
          ptx::mbar_arrive_expect_tx(kv_full + 8 * slot, Cfg::SLOT_BYTES);
          for (int part = 0; part < NPART; ++part)
            for (int at = 0; at < ATOMS; ++at)
              ptx::tma_load_2d(smem_ring + slot * Cfg::SLOT_BYTES + part * Cfg::PART_BYTES + at * ATT_TILE_BYTES, &tmap_qkv,
                               kv_full + 8 * slot, part * args.lo_col_off + which * D + kv_col[sl] + at * 64, kv_row[sl] + j * ATT_BKV);
          ++item;
        }
      };
      load(1, 0);
      for (int j = 0; j < n_kv; ++j) {
        if (j + 1 < n_kv) load(1, j + 1);
        load(2, j);
      }
      ++w;
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    // One elected thread issues (elect.sync lets ptxas emit the tcgen05 instructions without a per-instruction
    // leader-election loop); descriptors are advanced by compile-time constants in fully unrolled loops.
    if (ptx::elect_one()) {
      const uint32_t s_tmem = tmem_base + ATT_S_COL;
      const uint32_t o_tmem = tmem_base + Cfg::O_COL;
      const uint64_t q_desc = ptx::make_smem_desc_sw128(smem_q, 1024, 0);
      int item = 0;   // K/V ring position, running across work items
      int g = 0;      // KV blocks processed so far (all work items): phase counter of s_full / s_empty / p_full / o_full
      int w = 0;
      for (int it = blockIdx.x; it < args.n_items; it += gridDim.x) {
      int qt_unused, pair0_unused;
      bool packed;
      if (!att_decode<PACKED>(args, it, qt_unused, pair0_unused, packed)) continue;
      const int nslots = (PACKED && packed) ? args.pack : 1;
      const bool tl = tl0 && w == args.timeline_item;
      auto kv_len_mma = [&](int j) {  // keys of block j rounded up to the MMA granularity (16)
        int len = N - j * ATT_BKV;
        len = len > ATT_BKV ? ATT_BKV : len;
        return (len + 15) & ~15;
      };
      auto issue_s = [&](int j) {
        const uint32_t idesc = ptx::make_idesc(ATT_BQ, kv_len_mma(j), false, false, F16 ? 0u : 1u);
        if (nslots == 1) {   // ordinary item: straight-line issue (this is the path every full tile takes)
          const int slot = item % RING;
          ptx::mbar_wait(kv_full + 8 * slot, (item / RING) & 1, 11);
          ptx::tc_fence_after();
          const uint64_t k_desc = ptx::make_smem_desc_sw128(smem_ring + slot * Cfg::SLOT_BYTES, 1024, 0);
          // terms: (Qhi,Khi) [, (Qhi,Klo), (Qlo,Khi)]; K-major operands advance 32 B per 16-wide k step
#pragma unroll
          for (int t = 0; t < (SPLIT ? 3 : 1); ++t) {
            const uint64_t qa = ptx::desc_advance(q_desc, t == 2 ? Cfg::PART_BYTES : 0);
            const uint64_t ka = ptx::desc_advance(k_desc, t == 1 ? Cfg::PART_BYTES : 0);
            // k step = 16 columns: 32 B inside a swizzle atom, the next atom every 4 steps
#pragma unroll
            for (int k = 0; k < DH / 16; ++k)
              ptx::umma_bf16_ss(s_tmem, ptx::desc_advance(qa, (k >> 2) * ATT_TILE_BYTES + (k & 3) * 32),
                                ptx::desc_advance(ka, (k >> 2) * ATT_TILE_BYTES + (k & 3) * 32), idesc, (t | k) ? 1u : 0u);
          }
          ptx::umma_commit(kv_empty + 8 * slot);
          ++item;
        } else {
#pragma unroll 1
          for (int sl = 0; sl < nslots; ++sl) {   // packed item: one masked MMA group per slot, each against its own pair's K
            const int slot = item % RING;
            ptx::mbar_wait(kv_full + 8 * slot, (item / RING) & 1, 11);
            ptx::tc_fence_after();
            const uint64_t k_desc = ptx::make_smem_desc_sw128(smem_ring + slot * Cfg::SLOT_BYTES, 1024, 0);
            uint32_t lm[4];
            att_slot_mask(sl, nslots, lm);
#pragma unroll
            for (int t = 0; t < (SPLIT ? 3 : 1); ++t) {
              const uint64_t qa = ptx::desc_advance(q_desc, t == 2 ? Cfg::PART_BYTES : 0);
              const uint64_t ka = ptx::desc_advance(k_desc, t == 1 ? Cfg::PART_BYTES : 0);
#pragma unroll
              for (int k = 0; k < DH / 16; ++k)
                ptx::umma_bf16_ss_masked(s_tmem, ptx::desc_advance(qa, (k >> 2) * ATT_TILE_BYTES + (k & 3) * 32),
                                         ptx::desc_advance(ka, (k >> 2) * ATT_TILE_BYTES + (k & 3) * 32), idesc, (t | k) ? 1u : 0u, lm);
            }
            ptx::umma_commit(kv_empty + 8 * slot);
            ++item;
          }
        }
        ptx::umma_commit(s_full);
        att_stamp(args, tl, 1, j, 0);   // S_j issued
      };
      auto issue_pv = [&](int j) {
        // O accumulates across KV blocks in TMEM.
        // A = P in TMEM: 16 keys = 8 packed columns per step
        // B = V: MN-major [keys x DH]; 16 keys = two 8-row groups of 1024 B; at DH = 128 the second 64 columns are the
        // next swizzle atom (leading byte offset 16 KB)
        constexpr uint32_t idesc = ptx::make_idesc(ATT_BQ, DH, false, /*B = V is MN-major*/ true, F16 ? 0u : 1u);
        constexpr uint32_t v_lbo = DH == 64 ? 1024 : ATT_TILE_BYTES;
        const int ksteps = kv_len_mma(j) / 16;
        const uint32_t acc0 = j > 0 ? 1u : 0u;
        if (j == 0 && w > 0) {   // O still holds the previous work item until the softmax warps have read it out
          ptx::mbar_wait(o_empty, (w - 1) & 1, 17);
          ptx::tc_fence_after();
        }
        if (nslots == 1) {   // ordinary item: straight-line issue
          const int slot = item % RING;
          ptx::mbar_wait(kv_full + 8 * slot, (item / RING) & 1, 12);
          ptx::tc_fence_after();
          const uint64_t v_desc = ptx::make_smem_desc_sw128(smem_ring + slot * Cfg::SLOT_BYTES, 1024, v_lbo);
          // terms: (Phi,Vhi) [, (Phi,Vlo), (Plo,Vhi)]
#pragma unroll
          for (int t = 0; t < (SPLIT ? 3 : 1); ++t) {
            const uint32_t pa = tmem_base + Cfg::P_COL + (t == 2 ? 64 : 0);
            const uint64_t va = ptx::desc_advance(v_desc, t == 1 ? Cfg::PART_BYTES : 0);
            if (ksteps == ATT_BKV / 16) {
#pragma unroll
              for (int k = 0; k < ATT_BKV / 16; ++k)
                ptx::umma_bf16_ts(o_tmem, pa + k * 8, ptx::desc_advance(va, k * 2048), idesc, (t | k) ? 1u : acc0);
            } else {
#pragma unroll 1
              for (int k = 0; k < ksteps; ++k)
                ptx::umma_bf16_ts(o_tmem, pa + k * 8, ptx::desc_advance(va, k * 2048), idesc, (t | k) ? 1u : acc0);
            }
          }
          ptx::umma_commit(kv_empty + 8 * slot);
          ++item;
        } else {
#pragma unroll 1
          for (int sl = 0; sl < nslots; ++sl) {   // packed item: slot sl's rows of P against its own pair's V
            const int slot = item % RING;
            ptx::mbar_wait(kv_full + 8 * slot, (item / RING) & 1, 12);
            ptx::tc_fence_after();
            const uint64_t v_desc = ptx::make_smem_desc_sw128(smem_ring + slot * Cfg::SLOT_BYTES, 1024, v_lbo);
            uint32_t lm[4];
            att_slot_mask(sl, nslots, lm);
#pragma unroll
            for (int t = 0; t < (SPLIT ? 3 : 1); ++t) {
              const uint32_t pa = tmem_base + Cfg::P_COL + (t == 2 ? 64 : 0);
              const uint64_t va = ptx::desc_advance(v_desc, t == 1 ? Cfg::PART_BYTES : 0);
#pragma unroll 1
              for (int k = 0; k < ksteps; ++k)
                ptx::umma_bf16_ts_masked(o_tmem, pa + k * 8, ptx::desc_advance(va, k * 2048), idesc, (t | k) ? 1u : acc0, lm);
            }
            ptx::umma_commit(kv_empty + 8 * slot);
            ++item;
          }
        }
        ptx::umma_commit(o_full);
        att_stamp(args, tl, 1, j, 1);   // PV_j issued
      };
      ptx::mbar_wait(q_full, w & 1, 13);
      if (g > 0) ptx::mbar_wait(s_empty, (g - 1) & 1, 14);   // the previous item's last S has been read out of TMEM
      ptx::tc_fence_after();
      issue_s(0);
      if (n_kv == 1) ptx::umma_commit(q_empty);
      for (int j = 0; j < n_kv; ++j, ++g) {
        if (j + 1 < n_kv) {
          ptx::mbar_wait(s_empty, g & 1, 14);  // softmax has read S_j out of TMEM
          ptx::tc_fence_after();
          issue_s(j + 1);
          if (j + 2 == n_kv) ptx::umma_commit(q_empty);   // last S MMA of the item: Q tile reusable once it retires
        }
        ptx::mbar_wait(p_full, g & 1, 15);     // P_j in TMEM, O rescaled if needed
        ptx::tc_fence_after();
        issue_pv(j);
      }
      ++w;
      }
    }
   }
  } else {
    // ===================== softmax / output (warps 0..3) =====================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(Cfg::REGS_SOFTMAX));
    const int q = warp & 3;
    const int r = q * 32 + lane;  // query row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float sl2 = args.scale_log2;
    const uint64_t sl2_2 = ptx::dup_f32x2(sl2);
    int g = 0;                    // KV blocks processed so far (all work items): barrier phase counter
    int w = 0;
    for (int it = blockIdx.x; it < args.n_items; it += gridDim.x) {
    {
      int qt0, pair00;
      bool packed0;
      if (!att_decode<PACKED>(args, it, qt0, pair00, packed0)) continue;   // (decoded again for the epilogue: nothing of it stays live over the KV loop)
    }
    const bool tl = tl0 && w == args.timeline_item;
    float m_used = -INFINITY;     // the row maximum the exponentials are taken against
    float m_next = -INFINITY;     // a larger maximum seen in the previous block (lazy rescale pending)
    float l_run = 0.f;            // running row sum (same units as O in TMEM)

    for (int j = 0; j < n_kv; ++j, ++g) {
      int kv_len = N - j * ATT_BKV;
      kv_len = kv_len > ATT_BKV ? ATT_BKV : kv_len;
      const int nchunks = (((kv_len + 15) & ~15) + 31) >> 5;   // 32-column chunks the MMA produced
      att_stamp(args, tl && warp == 0, 0, j, 0);   // waiting for S_j
      ptx::mbar_wait(s_full, g & 1, 21);
      ptx::tc_fence_after();
      att_stamp(args, tl && warp == 0, 0, j, 1);   // S_j complete
      // ---- S_j -> registers (one pass), then hand the TMEM columns back to the MMA warp
      uint32_t s[4][32];
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < nchunks) ptx::tmem_ld_32x32b_x32(lane_addr + ATT_S_COL + c * 32, s[c]);
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < nchunks) ptx::tmem_ld_wait(s[c]);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(s_empty);
      att_stamp(args, tl && warp == 0, 0, j, 2);   // S_j in registers
      // ---- ragged last block only: columns beyond the sequence (and chunks the MMA never wrote) -> -inf,
      //      so the common path below carries no masks (exp2(-inf) = 0)
      if (kv_len < ATT_BKV) {
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (c * 32 + i >= kv_len) s[c][i] = 0xff800000u;
      }
      // ---- row maximum.  Block 0 needs it before any exponential (it sets the scale).  For the later blocks the
      // exponentials are taken against the maximum already in use and this block's maximum is computed inside the
      // same instruction stream (off the critical path): softmax is shift invariant and O / l live in fp32, so a
      // stale maximum costs nothing until a row exceeds it by 2^ATT_RESCALE_THRESHOLD -- then O and l are rescaled
      // before the NEXT block -- or by 2^ATT_REDO_THRESHOLD inside one block -- then this block is redone.
      auto row_max = [&]() {
        float mx4[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float m0 = fmaxf(__uint_as_float(s[c][0]), __uint_as_float(s[c][1]));
#pragma unroll
          for (int i = 2; i < 32; i += 2) m0 = fmaxf(fmaxf(m0, __uint_as_float(s[c][i])), __uint_as_float(s[c][i + 1]));
          mx4[c] = m0;
        }
        return fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      };
      if (j == 0) m_used = row_max();
      // ---- a maximum raised by the previous block: rescale l now, O once PV_{j-1} has completed
      float alpha = 1.0f;
      if (m_next > m_used) {
        alpha = ptx::ex2_approx((m_used - m_next) * sl2);
        m_used = m_next;
        l_run *= alpha;
      }
      att_stamp(args, tl && warp == 0, 0, j, 3);   // scale known
      auto rescale_o = [&](float a) {
#pragma unroll
        for (int c = 0; c < DH; c += 32) {
          uint32_t t[32];
          ptx::tmem_ld_32x32b_x32(lane_addr + Cfg::O_COL + c, t);
          ptx::tmem_ld_wait(t);
#pragma unroll
          for (int i = 0; i < 32; ++i) t[i] = __float_as_uint(__uint_as_float(t[i]) * a);
          ptx::tmem_st_32x32b_x32(lane_addr + Cfg::O_COL + c, t);
        }
      };
      if (j > 0) {
        ptx::mbar_wait(o_full, (g - 1) & 1, 20);   // PV_{j-1} done: the P columns are free, O is complete up to j-1
        ptx::tc_fence_after();
        att_stamp(args, tl && warp == 0, 0, j, 4); // PV_{j-1} complete
        if (__any_sync(0xffffffffu, alpha != 1.0f)) rescale_o(alpha);
      }
      // ---- p = exp2(s*sl2 - m*sl2) -> bf16 pairs -> TMEM columns P_COL + key/2 of this thread's lane
      // (the A operand of the PV MMA).  Optionally some pairs take the FMA-pipe polynomial instead of MUFU.EX2
      // (full blocks only: the ragged block carries -inf).
      uint64_t sum2[2];
      auto exp_chunks = [&](auto poly_tag) {
        constexpr bool POLY = decltype(poly_tag)::value;
        const uint64_t nm2 = ptx::dup_f32x2(-m_used * sl2);
        sum2[0] = 0ull;
        sum2[1] = 0ull;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c < nchunks) {
            uint32_t ph[16], pl[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const uint64_t a2 = ptx::fma_f32x2(ptx::pack_f32x2(__uint_as_float(s[c][2 * i]), __uint_as_float(s[c][2 * i + 1])), sl2_2, nm2);
              float e0, e1;
              if (POLY && ((POLY_MASK >> i) & 1u)) {
                ptx::ex2_poly_x2(a2, e0, e1);
              } else {
                float a0, a1;
                ptx::unpack_f32x2(a2, a0, a1);
                e0 = ptx::ex2_approx(a0);
                e1 = ptx::ex2_approx(a1);
              }
              sum2[i & 1] = ptx::add_f32x2(sum2[i & 1], ptx::pack_f32x2(e0, e1));
              ph[i] = ptx::pack_h2<F16>(e0, e1);
              if (SPLIT) pl[i] = ptx::pack_h2<F16>(e0 - ptx::round_h<F16>(e0), e1 - ptx::round_h<F16>(e1));
            }
            ptx::tmem_st_32x32b_x16(lane_addr + Cfg::P_COL + c * 16, ph);
            if (SPLIT) ptx::tmem_st_32x32b_x16(lane_addr + Cfg::P_COL + 64 + c * 16, pl);
          }
        }
      };
      auto run_exps = [&]() {
        if (!SPLIT && POLY_MASK != 0 && kv_len == ATT_BKV) exp_chunks(std::true_type{}); else exp_chunks(std::false_type{});
      };
      run_exps();
      if (j > 0 && !args.track_max) {
        float a0, a1, b0, b1;
        ptx::unpack_f32x2(sum2[0], a0, a1);
        ptx::unpack_f32x2(sum2[1], b0, b1);
        const float bsum = (a0 + a1) + (b0 + b1);
        // !(bsum <= T) also catches inf / NaN sums
        if (__any_sync(0xffffffffu, !(bsum <= (F16 ? ATT_SUM_TRIGGER_F16 : ATT_SUM_TRIGGER)))) {
          const float m_blk = row_max();
          const float m_new = fmaxf(m_used, m_blk);
          const float a = ptx::ex2_approx((m_used - m_new) * sl2);
          m_used = m_new;
          l_run *= a;
          rescale_o(a);
          run_exps();
        }
      } else if (j > 0) {
        const float excess = (row_max() - m_used) * sl2;       // independent of the exponentials above: overlaps them
        constexpr float REDO = F16 ? ATT_REDO_THRESHOLD_F16 : ATT_REDO_THRESHOLD;
        if (__any_sync(0xffffffffu, excess > REDO)) {
          // rare: a row jumped so far above the running maximum that exp2 may have overflowed -> raise the maximum
          // now (O is complete up to block j-1 and may be rescaled here) and redo this block's exponentials
          const float m_new = excess > REDO ? m_used + excess / sl2 : m_used;
          const float a = ptx::ex2_approx((m_used - m_new) * sl2);
          m_used = m_new;
          l_run *= a;
          rescale_o(a);
          run_exps();
        } else if (excess > ATT_RESCALE_THRESHOLD) {
          m_next = m_used + excess / sl2;                        // applied before the next block
        }
      }
      {
        float a0, a1, b0, b1;
        ptx::unpack_f32x2(sum2[0], a0, a1);
        ptx::unpack_f32x2(sum2[1], b0, b1);
        l_run += (a0 + a1) + (b0 + b1);
      }
      att_stamp(args, tl && warp == 0, 0, j, 5);   // exponentials issued
      ptx::tmem_st_wait();             // P (and a rescaled O) are in TMEM
      ptx::tc_fence_before();          // ... and ordered before the MMA that reads / accumulates on them
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(p_full);
      att_stamp(args, tl && warp == 0, 0, j, 6);   // P_j handed to the MMA warp
    }
    // ---- epilogue: ctx = O / l
    ptx::mbar_wait(o_full, (g - 1) & 1, 22);
    ptx::tc_fence_after();
    const float inv = 1.0f / l_run;
    // this thread's row: tile row r of an ordinary item; in a packed item row (r % slot_rows) of the tail of pair0 + r / slot_rows
    int qt, pair0;
    bool packed;
    att_decode<PACKED>(args, it, qt, pair0, packed);
    int my_pair = pair0, row_in_tile = r, slot_rows = ATT_BQ;
    if (PACKED && packed) {
      slot_rows = ATT_BQ / args.pack;
      const int sl = r / slot_rows;
      row_in_tile = r - sl * slot_rows;
      my_pair = pair0 + sl;
    }
    const bool pair_ok = my_pair < args.n_pairs;
    const int b = my_pair / args.heads, h = my_pair - b * args.heads;
    const int row_base = b * N;
    const int qrow = qt * ATT_BQ + row_in_tile;
    if (args.lse2 != nullptr && pair_ok) {   // pad rows get +inf: the backward turns that into P = 0 without a bounds test
      float* lrow = args.lse2 + static_cast<long long>(my_pair) * (args.n_qtiles * ATT_BQ);
      lrow[qrow] = qrow < N ? m_used * sl2 + log2f(l_run) : INFINITY;
      for (int k = slot_rows; k < ATT_BQ; k += slot_rows) lrow[qrow + k] = INFINITY;   // packed item: the rest of the pad rows
    }
    __nv_bfloat16* o = args.out + static_cast<long long>(row_base + qrow) * args.ldo + h * DH;
    // 64 columns of O (64 registers) per pass: all 128 columns of head_dim 128 at once would spill
#pragma unroll
    for (int ps = 0; ps < DH / 64; ++ps) {
      uint32_t t[2][32];
#pragma unroll
      for (int c = 0; c < 2; ++c) ptx::tmem_ld_32x32b_x32(lane_addr + Cfg::O_COL + ps * 64 + c * 32, t[c]);
#pragma unroll
      for (int c = 0; c < 2; ++c) ptx::tmem_ld_wait(t[c]);
      if (ps == DH / 64 - 1) {
        // O is in registers: the MMA warp may start accumulating the next work item into the same columns
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(o_empty);
      }
      if (qrow < N && pair_ok) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
#pragma unroll
          for (int q4 = 0; q4 < 4; ++q4) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(t[c][8 * q4 + i]) * inv;
            reinterpret_cast<uint4*>(o + ps * 64 + c * 32)[q4] = make_uint4(ptx::pack_h2<F16>(v[0], v[1]), ptx::pack_h2<F16>(v[2], v[3]),
                                                                            ptx::pack_h2<F16>(v[4], v[5]), ptx::pack_h2<F16>(v[6], v[7]));
            if (SPLIT) {
              float lo[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) lo[i] = v[i] - ptx::round_h<F16>(v[i]);
              reinterpret_cast<uint4*>(o + args.out_lo_off + ps * 64 + c * 32)[q4] =
                  make_uint4(ptx::pack_h2<F16>(lo[0], lo[1]), ptx::pack_h2<F16>(lo[2], lo[3]), ptx::pack_h2<F16>(lo[4], lo[5]),
                             ptx::pack_h2<F16>(lo[6], lo[7]));
            }
          }
        }
      }
    }
    ++w;
    }   // work items
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (tl0 && threadIdx.x == 0) args.timeline[((blockIdx.x * 2 + 0) * ATT_TL_BLOCKS + 15) * ATT_TL_EVENTS + 7] = clock64();   // CTA end
  if (warp == 5) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace vitocm
