// Forward attention, "quad" form: FOUR independent softmax pipelines per SM (one 640-thread CTA per SM), 64-key blocks.
// Replaces SSS/dino/vision_transformer.py:83-87 like attention_sm100.cuh, for the FULL 128-row query tiles of 16-bit engines
// AND, as its first items, for the ragged query tails: the tails of `pack` = 2 (image, head) pairs share one 128-row tile, one masked
// MMA group per pair (the packed items of attention_sm100.cuh, here on 64-key blocks; two pairs, not four: a block's K and V tiles of
// two pairs stream through the five-slot ring without a stall, those of four do not -- measured 4 x slower per item).
//
// Why: the exponentials bound this kernel (MUFU: 16 ex2 / clk / SM), and ONE warp per scheduler can only issue a MUFU every
// ~14 clk against the unit's 8 (profiles/r01_attention_phased_exps.txt).  The two co-resident CTAs of attn_fwd_tcgen05_kernel
// put two softmax warps on every scheduler, so the unit is only saturated while BOTH are inside their exponentials, and nothing
// hides the rest of a block (S wait, TMEM -> registers, bookkeeping, hand-over: ~1 150 of ~3 150 clk per 128-key block, XU 45 %
// in ncu).  Four pipelines put four softmax warps on every scheduler: while one or two are in the latency-bound part of their
// block the others keep the MUFU busy.  What makes four fit:
//   * 64-key blocks and P written OVER S: a pipeline owns 128 TMEM columns (S 64 fp32 columns, the packed 16-bit P over its
//     first 32; O 64) -- 4 x 128 = 512.  QK_{j+1} is only issued after PV_j (same issuing thread, the tensor pipe executes in
//     order), so a pipeline's MMAs and exponentials strictly alternate; the other three pipelines fill the gaps;
//   * a softmax thread holds 64 logits instead of 128: 104 registers (16 warps x 104 + 4 control warps x 48 <= 640 x 96);
//   * one control warp per pipeline whose elected thread is TMA producer AND MMA issuer (in-order anyway): K / V stream
//     through a private ring of five 8 KB tiles, Q (16 KB) is re-loaded as soon as the item's last S has been produced.
// Per thread the arithmetic is the one of attn_fwd_tcgen05_kernel with track_max = 0, one 32-key chunk at a time (the first chunk
// fixes the row maximum, every later chunk is checked through its row sum and redone against a larger maximum when it trips).
#pragma once
#include "attention_sm100.cuh"

namespace vitocm {

constexpr int AQ_PIPES = 4;
constexpr int AQ_BKV = 64;
constexpr int AQ_RING = 5;                            // K / V tiles in flight per pipeline
constexpr int AQ_TILE_BYTES = AQ_BKV * ATT_DH * 2;    // 8 KB: one [64 keys x 64] tile
constexpr int AQ_Q_BYTES = ATT_BQ * ATT_DH * 2;       // 16 KB
constexpr int AQ_THREADS = (4 * AQ_PIPES + 4) * 32;   // 16 softmax warps + 4 control warps
constexpr int AQ_PIPE_SMEM = AQ_Q_BYTES + AQ_RING * AQ_TILE_BYTES;
constexpr int AQ_PIPE_BARS = 128;
constexpr int AQ_SMEM_BYTES = AQ_PIPES * (AQ_PIPE_SMEM + AQ_PIPE_BARS) + 64 + 1024 /*alignment slack*/;
constexpr int AQ_REGS_SOFTMAX = 104;
constexpr int AQ_REGS_CTRL = 64;
static_assert(16 * AQ_REGS_SOFTMAX + 4 * AQ_REGS_CTRL <= 20 * 96, "quad attention: setmaxnreg budgets exceed the launch allocation");
static_assert(AQ_SMEM_BYTES <= 227 * 1024, "quad attention: shared memory");
constexpr int AQ_S_COL = 0;     // S: 64 fp32 columns; P (packed pairs, 32 columns) over its first half
constexpr int AQ_O_COL = 64;    // O: 64 fp32 columns

// work item -> (first pair, query tile, pairs sharing the tile).  Without tail items (group_items == 0): query tile fastest, then the
// pair.  With them: groups of `pack` consecutive pairs = pack x n_fullq full tiles followed by the ONE tile their ragged tails
// share, so that the tail runs while its pairs' K / V are hot in L2 (tails first or last re-read every K / V from HBM: 1.5 GB per
// launch at the bench's size).  Pairs beyond the batch (last group) are clamped by the callers: computed, not stored.
__device__ __forceinline__ void aq_decode(const AttnArgs& a, int it, int& pair0, int& qt, int& nslots) {
  if (a.group_items == 0) {
    pair0 = it / a.n_fullq;
    qt = it - pair0 * a.n_fullq;
    nslots = 1;
    return;
  }
  const int g = it / a.group_items, r = it - g * a.group_items;
  if (r < a.pack * a.n_fullq) {
    const int pi = r / a.n_fullq;
    pair0 = g * a.pack + pi;
    qt = r - pi * a.n_fullq;
    nslots = 1;
  } else {
    pair0 = g * a.pack;
    qt = a.n_fullq;
    nslots = a.pack;
  }
}
// disable-output-lane mask of slot SL of NS equal lane groups as compile-time constants (run-time masks cost the issuing thread four
// R2UR round trips per MMA: ~150 clk per masked MMA against ~40 -- profiles/r02 timeline of a tail item)
template <int NS, int SL>
__device__ __forceinline__ void aq_slot_mask(uint32_t (&m)[4]) {
#pragma unroll
  for (int w = 0; w < 4; ++w) m[w] = ((NS == 4 ? w : (NS == 2 ? (w >> 1) : 0)) == SL) ? 0u : 0xffffffffu;
}

// TL: clock stamps of tools/attn_quad_timeline.py (a separate instantiation: the stamps cost registers)
// VARLEN: items come from AttnArgs::vitems (images of different sizes packed back to back, see att_vdecode)
template <bool F16, bool TL = false, bool VARLEN = false>
__global__ void __launch_bounds__(AQ_THREADS, 1)
attn_fwd_quad_kernel(const __grid_constant__ CUtensorMap tmap_q /*box 64 x 128*/, const __grid_constant__ CUtensorMap tmap_kv /*box 64 x 64*/,
                     const __grid_constant__ CUtensorMap tmap_q32 /*box 64 x 32: the query slots of packed tail items*/, const AttnArgs args) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t smem = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bars0 = smem + AQ_PIPES * AQ_PIPE_SMEM;
  const uint32_t tmem_ptr_smem = bars0 + AQ_PIPES * AQ_PIPE_BARS;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int N = args.n_tokens;
  const int D = args.embed_dim;
  const int n_kv = (N + AQ_BKV - 1) / AQ_BKV;
  const int p = warp < 4 * AQ_PIPES ? (warp >> 2) : (warp - 4 * AQ_PIPES);   // pipeline of this warp
  const uint32_t smem_q = smem + p * AQ_PIPE_SMEM;
  const uint32_t smem_ring = smem_q + AQ_Q_BYTES;
  const uint32_t bars = bars0 + p * AQ_PIPE_BARS;
  const uint32_t q_full = bars;            // Q tile landed
  const uint32_t s_full = bars + 8;        // S_j complete in TMEM (all earlier MMAs of the pipeline retired)
  const uint32_t p_full = bars + 16;       // P_j in TMEM (4 warps)
  const uint32_t o_full = bars + 24;       // last PV of the item retired
  const uint32_t o_empty = bars + 32;      // O of the finished item has been read out (4 warps)
  const uint32_t kv_full = bars + 40;      // [AQ_RING]
  const uint32_t kv_empty = bars + 80;     // [AQ_RING]
  static_assert(80 + 8 * AQ_RING <= AQ_PIPE_BARS, "quad attention: barrier block");

  if (warp == 4 * AQ_PIPES && lane == 0) {
    ptx::prefetch_tmap(&tmap_q);
    ptx::prefetch_tmap(&tmap_kv);
    ptx::prefetch_tmap(&tmap_q32);
    for (int pp = 0; pp < AQ_PIPES; ++pp) {
      const uint32_t b = bars0 + pp * AQ_PIPE_BARS;
      ptx::mbar_init(b, 1);
      ptx::mbar_init(b + 8, 1);
      ptx::mbar_init(b + 16, 4);
      ptx::mbar_init(b + 24, 1);
      ptx::mbar_init(b + 32, 4);
      for (int i = 0; i < AQ_RING; ++i) {
        ptx::mbar_init(b + 40 + 8 * i, 1);
        ptx::mbar_init(b + 80 + 8 * i, 1);
      }
    }
    ptx::fence_barrier_init();
  }
  if (warp == 4 * AQ_PIPES + 1) {
    ptx::tmem_alloc(tmem_ptr_smem, 512);
    ptx::tmem_relinquish();
  }
  if (warp == 4 * AQ_PIPES + 2 && lane == 0 && args.stagger_clk > 0) {   // start stagger (AttnArgs::stagger_clk)
    const long long wait_clk = static_cast<long long>(args.stagger_clk) * blockIdx.x / gridDim.x;
    const long long t0 = clock64();
    while (clock64() - t0 < wait_clk) {}
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = ptx::lds_u32(tmem_ptr_smem) + static_cast<uint32_t>(p * 128);

  // work items of this pipeline (aq_decode); the four pipelines of a CTA take consecutive items, so they read one pair's K / V through
  // L2 at about the same time
  const int first = static_cast<int>(blockIdx.x) * AQ_PIPES + p;
  const int stride = static_cast<int>(gridDim.x) * AQ_PIPES;

  if (warp >= 4 * AQ_PIPES) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(AQ_REGS_CTRL));
    // ===================== control warp: TMA producer + MMA issuer of pipeline p =====================
    if (ptx::elect_one()) {
      const uint32_t s_tmem = tmem_base + AQ_S_COL, o_tmem = tmem_base + AQ_O_COL;
      const uint64_t q_desc = ptx::make_smem_desc_sw128(smem_q, 1024, 0);
      int Ni = N;   // tokens of the current item's image (VARLEN: per item)
      auto kv_len_mma = [&](int j) {   // keys of block j rounded up to the MMA granularity (16)
        int len = Ni - j * AQ_BKV;
        len = len > AQ_BKV ? AQ_BKV : len;
        return (len + 15) & ~15;
      };
      // pair of slot s (slots beyond the batch repeat the last pair: their rows are computed and dropped)
      auto clamp_pair = [&](int pr) { return pr < args.n_pairs ? pr : args.n_pairs - 1; };
      auto load_q = [&](int it) {
        int pair0, qt, ns;
        if constexpr (VARLEN) {
          int row0, n, h0;
          att_vdecode(args, it, row0, n, qt, h0, ns);
          ptx::mbar_arrive_expect_tx(q_full, AQ_Q_BYTES);
          if (ns == 1) {
            ptx::tma_load_2d(smem_q, &tmap_q, q_full, h0 * ATT_DH, row0 + qt * ATT_BQ);
          } else {
            const int per = 4 / ns;
            for (int u = 0; u < 4; ++u)
              ptx::tma_load_2d(smem_q + u * 4096, &tmap_q32, q_full, min(h0 + u / per, args.heads - 1) * ATT_DH, row0 + qt * ATT_BQ + (u % per) * 32);
          }
          return;
        }
        aq_decode(args, it, pair0, qt, ns);
        ptx::mbar_arrive_expect_tx(q_full, AQ_Q_BYTES);
        if (ns == 1) {
          const int pair = clamp_pair(pair0);
          const int b = pair / args.heads, h = pair - b * args.heads;
          ptx::tma_load_2d(smem_q, &tmap_q, q_full, h * ATT_DH, b * N + qt * ATT_BQ);
        } else {   // four 32-row boxes; slot s owns tile rows [s * 128 / pack, (s + 1) * 128 / pack) = the first rows of its pair's tail
          const int per = 4 / ns;
          for (int u = 0; u < 4; ++u) {
            const int pr = clamp_pair(pair0 + u / per);
            const int b = pr / args.heads, h = pr - b * args.heads;
            ptx::tma_load_2d(smem_q + u * 4096, &tmap_q32, q_full, h * ATT_DH, b * N + qt * ATT_BQ + (u % per) * 32);
          }
        }
      };
      // K / V stream in consumption order (per block: K of every slot, then V of every slot), running across the items of this pipeline
      int loaded = 0, used = 0;          // tiles requested / handed to an MMA
      int l_it = first, l_j = 0, l_which = 1, l_sl = 0, l_ns = 1;   // next tile to request: item, block, 1 = K / 2 = V, slot; slots of the item
      int l_col = 0, l_row = 0, l_nkv = n_kv;
      auto set_load_coords = [&]() {
        if (l_it < args.n_items) {
          int pair0, qt;
          if constexpr (VARLEN) {
            int n, h0;
            att_vdecode(args, l_it, l_row, n, qt, h0, l_ns);
            l_col = min(h0 + l_sl, args.heads - 1) * ATT_DH;
            l_nkv = (n + AQ_BKV - 1) / AQ_BKV;
            return;
          }
          aq_decode(args, l_it, pair0, qt, l_ns);
          const int pr = clamp_pair(pair0 + l_sl);
          const int b = pr / args.heads;
          l_col = (pr - b * args.heads) * ATT_DH;
          l_row = b * N;
        }
      };
      set_load_coords();
      auto fill = [&]() {
        while (loaded - used < AQ_RING && l_it < args.n_items) {
          const int slot = loaded % AQ_RING;
          if (loaded >= AQ_RING) ptx::mbar_wait(kv_empty + 8 * slot, ((loaded / AQ_RING) - 1) & 1, 50);   // the MMA that read it retired
          ptx::mbar_arrive_expect_tx(kv_full + 8 * slot, AQ_TILE_BYTES);
          ptx::tma_load_2d(smem_ring + slot * AQ_TILE_BYTES, &tmap_kv, kv_full + 8 * slot, l_which * D + l_col, l_row + l_j * AQ_BKV);
          ++loaded;
          bool recode = l_ns > 1;
          if (++l_sl == l_ns) {
            l_sl = 0;
            if (l_which == 1) {
              l_which = 2;
            } else {
              l_which = 1;
              if (++l_j == l_nkv) { l_j = 0; l_it += stride; recode = true; }
            }
          }
          if (recode) set_load_coords();
        }
      };
      if (first < args.n_items) load_q(first);
      fill();
      // S_j = Q K_j^T into the columns that held P_{j-1}: it is issued right BEHIND PV_{j-1} (the tensor pipe executes in order, so
      // PV_{j-1} has read P before S_j lands on it), never behind a wait for PV_{j-1} to retire -- ring refills come after the issue
      auto issue_s = [&](int j, int nslots) {
        const uint32_t idesc = ptx::make_idesc(ATT_BQ, kv_len_mma(j), false, false, F16 ? 0u : 1u);
        if (nslots == 1) {
          const int slot = used % AQ_RING;
          ptx::mbar_wait(kv_full + 8 * slot, (used / AQ_RING) & 1, 52);
          ptx::tc_fence_after();
          const uint64_t k_desc = ptx::make_smem_desc_sw128(smem_ring + slot * AQ_TILE_BYTES, 1024, 0);
#pragma unroll
          for (int k = 0; k < ATT_DH / 16; ++k)
            ptx::umma_bf16_ss(s_tmem, ptx::desc_advance(q_desc, k * 32), ptx::desc_advance(k_desc, k * 32), idesc, k ? 1u : 0u);
          ptx::umma_commit(kv_empty + 8 * slot);
          ++used;
        } else {   // packed item: one masked MMA group per slot, each against its own pair's K
          auto slot_s = [&](auto ns_tag, auto sl_tag) {
            if (loaded <= used) fill();   // (pack = 4: a block's eight tiles do not fit the ring, requests continue between the groups)
            const int slot = used % AQ_RING;
            ptx::mbar_wait(kv_full + 8 * slot, (used / AQ_RING) & 1, 56);
            ptx::tc_fence_after();
            const uint64_t k_desc = ptx::make_smem_desc_sw128(smem_ring + slot * AQ_TILE_BYTES, 1024, 0);
            uint32_t lm[4];
            aq_slot_mask<decltype(ns_tag)::value, decltype(sl_tag)::value>(lm);
#pragma unroll
            for (int k = 0; k < ATT_DH / 16; ++k)
              ptx::umma_bf16_ss_masked(s_tmem, ptx::desc_advance(q_desc, k * 32), ptx::desc_advance(k_desc, k * 32), idesc, k ? 1u : 0u, lm);
            ptx::umma_commit(kv_empty + 8 * slot);
            ++used;
          };
          using I0 = std::integral_constant<int, 0>; using I1 = std::integral_constant<int, 1>;
          using I2 = std::integral_constant<int, 2>; using I3 = std::integral_constant<int, 3>; using I4 = std::integral_constant<int, 4>;
          if (nslots == 2) { slot_s(I2{}, I0{}); slot_s(I2{}, I1{}); }
          else { slot_s(I4{}, I0{}); slot_s(I4{}, I1{}); slot_s(I4{}, I2{}); slot_s(I4{}, I3{}); }
        }
        ptx::umma_commit(s_full);
      };
      int g = 0;   // KV blocks so far (all items): phase of s_full / p_full
      int w = 0;   // items so far: phase of q_full / o_full / o_empty
      for (int it = first; it < args.n_items; it += stride, ++w) {
        const bool tl = TL && args.timeline != nullptr && blockIdx.x == 0 && p < 2 && w == args.timeline_item;
        int nslots, pair0_unused, qt_unused, nkv = n_kv;
        if constexpr (VARLEN) {
          int r0_unused, h0_unused;
          att_vdecode(args, it, r0_unused, Ni, qt_unused, h0_unused, nslots);
          nkv = (Ni + AQ_BKV - 1) / AQ_BKV;
        } else {
        aq_decode(args, it, pair0_unused, qt_unused, nslots);
        }
        ptx::mbar_wait(q_full, w & 1, 51);
        issue_s(0, nslots);
        if constexpr (TL) att_stamp(args, tl, 1, 0, 0, p);   // S_0 issued
        for (int j = 0; j < nkv; ++j, ++g) {
          fill();
          constexpr uint32_t idesc_pv = ptx::make_idesc(ATT_BQ, ATT_DH, false, /*B = V is MN-major*/ true, F16 ? 0u : 1u);
          const int ksteps = kv_len_mma(j) / 16;
          const uint32_t acc0 = j > 0 ? 1u : 0u;
          if (nslots == 1 && args.ctrl_hoist) {
            // Everything PV_j and S_{j+1} need is prepared BEFORE the wait for P_j: the control warp shares its scheduler with four
            // softmax warps, so every instruction between "P_j seen" and the last MMA costs ~5 clk of the pipeline's serial chain
            // (descriptor arithmetic + operand-landed checks behind the wait: 850 clk from P_j to S_{j+1} issued, of ~3 250 per block)
            const bool more = j + 1 < nkv;
            const int slot_v = used % AQ_RING, slot_k = (used + 1) % AQ_RING;
            ptx::mbar_wait(kv_full + 8 * slot_v, (used / AQ_RING) & 1, 55);
            if (more) ptx::mbar_wait(kv_full + 8 * slot_k, ((used + 1) / AQ_RING) & 1, 52);
            const uint64_t v_desc = ptx::make_smem_desc_sw128(smem_ring + slot_v * AQ_TILE_BYTES, 1024, 1024);
            const uint64_t k_desc = ptx::make_smem_desc_sw128(smem_ring + slot_k * AQ_TILE_BYTES, 1024, 0);
            const uint32_t idesc_s = ptx::make_idesc(ATT_BQ, kv_len_mma(more ? j + 1 : j), false, false, F16 ? 0u : 1u);
            const uint32_t bar_v = kv_empty + 8 * slot_v, bar_k = kv_empty + 8 * slot_k;
            if (j == 0 && w > 0) ptx::mbar_wait(o_empty, (w - 1) & 1, 54);   // O still holds the previous item until its rows have been read out
            // ---- O += P_j V_j
            ptx::mbar_wait(p_full, g & 1, 53);
            ptx::tc_fence_after();
            if constexpr (TL) att_stamp(args, tl, 1, j, 1, p);   // P_j seen
            if (ksteps == AQ_BKV / 16) {
#pragma unroll
              for (int k = 0; k < AQ_BKV / 16; ++k)
                ptx::umma_bf16_ts(o_tmem, s_tmem + k * 8, ptx::desc_advance(v_desc, k * 2048), idesc_pv, k ? 1u : acc0);
            } else {
#pragma unroll 1
              for (int k = 0; k < ksteps; ++k)
                ptx::umma_bf16_ts(o_tmem, s_tmem + k * 8, ptx::desc_advance(v_desc, k * 2048), idesc_pv, k ? 1u : acc0);
            }
            ptx::umma_commit(bar_v);
            if constexpr (TL) att_stamp(args, tl, 1, j, 2, p);   // PV_j issued
            if (more) {
              // ---- S_{j+1} = Q K_{j+1}^T right behind it
#pragma unroll
              for (int k = 0; k < ATT_DH / 16; ++k)
                ptx::umma_bf16_ss(s_tmem, ptx::desc_advance(q_desc, k * 32), ptx::desc_advance(k_desc, k * 32), idesc_s, k ? 1u : 0u);
              ptx::umma_commit(bar_k);
              ptx::umma_commit(s_full);
              used += 2;
              if constexpr (TL) att_stamp(args, tl, 1, j + 1, 0, p);   // S_{j+1} issued
            } else {
              ptx::umma_commit(o_full);
              ++used;
              if (it + stride < args.n_items) load_q(it + stride);   // P_last exists => every S of the item was produced: Q is free
            }
            continue;
          }
          // ---- packed tail item: every slot's P rows against its own pair's V, then the next S per slot
          ptx::mbar_wait(p_full, g & 1, 53);
          ptx::tc_fence_after();
          if constexpr (TL) att_stamp(args, tl, 1, j, 1, p);   // P_j seen
          if (j == 0 && w > 0) {   // O still holds the previous item until its rows have been read out
            ptx::mbar_wait(o_empty, (w - 1) & 1, 54);
            ptx::tc_fence_after();
          }
          if (nslots == 1) {
            const int slot = used % AQ_RING;
            ptx::mbar_wait(kv_full + 8 * slot, (used / AQ_RING) & 1, 55);
            ptx::tc_fence_after();
            const uint64_t v_desc = ptx::make_smem_desc_sw128(smem_ring + slot * AQ_TILE_BYTES, 1024, 1024);
#pragma unroll 1
            for (int k = 0; k < ksteps; ++k)
              ptx::umma_bf16_ts(o_tmem, s_tmem + k * 8, ptx::desc_advance(v_desc, k * 2048), idesc_pv, k ? 1u : acc0);
            ptx::umma_commit(kv_empty + 8 * slot);
            ++used;
            if (j == nkv - 1) ptx::umma_commit(o_full);
          } else {
            auto slot_pv = [&](auto ns_tag, auto sl_tag) {
              if (loaded <= used) fill();
              const int slot = used % AQ_RING;
              ptx::mbar_wait(kv_full + 8 * slot, (used / AQ_RING) & 1, 57);
              ptx::tc_fence_after();
              const uint64_t v_desc = ptx::make_smem_desc_sw128(smem_ring + slot * AQ_TILE_BYTES, 1024, 1024);
              uint32_t lm[4];
              aq_slot_mask<decltype(ns_tag)::value, decltype(sl_tag)::value>(lm);
              if (ksteps == AQ_BKV / 16) {
#pragma unroll
                for (int k = 0; k < AQ_BKV / 16; ++k)
                  ptx::umma_bf16_ts_masked(o_tmem, s_tmem + k * 8, ptx::desc_advance(v_desc, k * 2048), idesc_pv, k ? 1u : acc0, lm);
              } else {
#pragma unroll 1
                for (int k = 0; k < ksteps; ++k)
                  ptx::umma_bf16_ts_masked(o_tmem, s_tmem + k * 8, ptx::desc_advance(v_desc, k * 2048), idesc_pv, k ? 1u : acc0, lm);
              }
              ptx::umma_commit(kv_empty + 8 * slot);
              ++used;
            };
            using I0 = std::integral_constant<int, 0>; using I1 = std::integral_constant<int, 1>;
            using I2 = std::integral_constant<int, 2>; using I3 = std::integral_constant<int, 3>; using I4 = std::integral_constant<int, 4>;
            if (nslots == 2) { slot_pv(I2{}, I0{}); slot_pv(I2{}, I1{}); }
            else { slot_pv(I4{}, I0{}); slot_pv(I4{}, I1{}); slot_pv(I4{}, I2{}); slot_pv(I4{}, I3{}); }
            if (j == nkv - 1) ptx::umma_commit(o_full);
          }
          if constexpr (TL) att_stamp(args, tl, 1, j, 2, p);   // PV_j issued
          if (j + 1 < nkv) {
            issue_s(j + 1, nslots);
            if constexpr (TL) att_stamp(args, tl, 1, j + 1, 0, p);   // S_{j+1} issued
          } else if (it + stride < args.n_items) {
            load_q(it + stride);   // P_last exists => every S of the item was produced: Q is free
          }
        }
      }
      // (every tile requested by fill() has been consumed: requests stop with the last item's last V)
    }
  } else {
    // ===================== softmax / output: warps 4p .. 4p+3 =====================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(AQ_REGS_SOFTMAX));
    const int q = warp & 3;
    const int r = q * 32 + lane;   // query row inside the tile == TMEM lane
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float sl2 = args.scale_log2;
    const uint64_t sl2_2 = ptx::dup_f32x2(sl2);
    int g = 0, w = 0;
    for (int it = first; it < args.n_items; it += stride, ++w) {
      const bool tl = TL && args.timeline != nullptr && blockIdx.x == 0 && p < 2 && q == 0 && lane == 0 && w == args.timeline_item;
      float m_used = -INFINITY;   // the row maximum the exponentials are taken against
      float l_run = 0.f;          // running row sum (same units as O in TMEM)
      int Ni = N, nkv = n_kv;
      bool votes = true;   // VARLEN: only rows of the item's own image and heads vote on a redo (see attn_fwd_tcgen05_kernel)
      if constexpr (VARLEN) {
        int r0_unused, vqt, vh0, vns;
        att_vdecode(args, it, r0_unused, Ni, vqt, vh0, vns);
        nkv = (Ni + AQ_BKV - 1) / AQ_BKV;
        const int slot_rows = ATT_BQ / vns, sl = r / slot_rows;
        votes = vh0 + sl < args.heads && vqt * ATT_BQ + (r - sl * slot_rows) < Ni;
      }
      for (int j = 0; j < nkv; ++j, ++g) {
        int kv_len = Ni - j * AQ_BKV;
        kv_len = kv_len > AQ_BKV ? AQ_BKV : kv_len;
        const int nchunks = (((kv_len + 15) & ~15) + 31) >> 5;   // 32-column chunks the MMA produced
        if constexpr (TL) att_stamp(args, tl, 0, j, 0, p);     // waiting for S_j
        ptx::mbar_wait(s_full, g & 1, 60);   // S_j complete; PV_{j-1} retired too: O is complete up to block j-1, the P columns are free
        ptx::tc_fence_after();
        if constexpr (TL) att_stamp(args, tl, 0, j, 1, p);     // S_j complete
        // One 32-key chunk at a time (32 logits live, not 64: the kernel runs at 104 registers per softmax thread).  The chunk's P goes
        // into columns S_COL + 16 c ... of the lane: over logits this thread has already consumed (chunk 1's logits sit in columns
        // 32 .. 63, untouched by P).  Reference maximum = the maximum of chunk 0 of block 0; EVERY other chunk is checked through its
        // row sum: a stale maximum is exact (softmax is shift invariant, O and l accumulate in fp32) until an exponential overflows
        // the 16-bit P format, and only a chunk whose sum trips the trigger pays for its maximum, the rescale of O / l / the block's
        // earlier P and a second pass of exponentials.
        float bsum = 0.f;   // this block's row sum
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          if (c < nchunks) {
            uint32_t s[32];
            ptx::tmem_ld_32x32b_x32(lane_addr + AQ_S_COL + c * 32, s);
            ptx::tmem_ld_wait(s);
            if constexpr (TL) att_stamp(args, tl, 0, j, 2 + 2 * c, p);   // chunk c in registers
            if (kv_len < AQ_BKV) {   // ragged last block: columns beyond the sequence -> -inf (exp2(-inf) = 0)
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c * 32 + i >= kv_len) s[i] = 0xff800000u;
            }
            auto chunk_max = [&]() {
              float m0 = fmaxf(__uint_as_float(s[0]), __uint_as_float(s[1]));
#pragma unroll
              for (int i = 2; i < 32; i += 2) m0 = fmaxf(fmaxf(m0, __uint_as_float(s[i])), __uint_as_float(s[i + 1]));
              return m0;
            };
            if (j == 0 && c == 0) m_used = chunk_max();
            float csum;
            auto run_exps = [&]() {   // p = exp2(s*sl2 - m*sl2) -> 16-bit pairs -> TMEM (the A operand of the PV MMA)
              const uint64_t nm2 = ptx::dup_f32x2(-m_used * sl2);
              uint64_t sum2[2] = {0ull, 0ull};
              uint32_t ph[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const uint64_t a2 = ptx::fma_f32x2(ptx::pack_f32x2(__uint_as_float(s[2 * i]), __uint_as_float(s[2 * i + 1])), sl2_2, nm2);
                float a0, a1;
                ptx::unpack_f32x2(a2, a0, a1);
                const float e0 = ptx::ex2_approx(a0), e1 = ptx::ex2_approx(a1);
                sum2[i & 1] = ptx::add_f32x2(sum2[i & 1], ptx::pack_f32x2(e0, e1));
                ph[i] = ptx::pack_h2<F16>(e0, e1);
              }
              ptx::tmem_st_32x32b_x16(lane_addr + AQ_S_COL + c * 16, ph);
              float a0, a1, b0, b1;
              ptx::unpack_f32x2(sum2[0], a0, a1);
              ptx::unpack_f32x2(sum2[1], b0, b1);
              csum = (a0 + a1) + (b0 + b1);
            };
            run_exps();
            // !(csum <= T) also catches inf / NaN sums
            if ((j > 0 || c > 0) && __any_sync(0xffffffffu, votes && !(csum <= (F16 ? ATT_SUM_TRIGGER_F16 : ATT_SUM_TRIGGER)))) {
              const float m_new = fmaxf(m_used, chunk_max());
              const float a = ptx::ex2_approx((m_used - m_new) * sl2);
              m_used = m_new;
              l_run *= a;
              bsum *= a;
              if (j > 0) {   // O holds the blocks before this one (PV_{j-1} retired before S_j completed): 8 columns at a time
#pragma unroll 1
                for (int oc = 0; oc < ATT_DH; oc += 8) {
                  uint32_t t[8];
                  ptx::tmem_ld_32x32b_x8(lane_addr + AQ_O_COL + oc, t);
                  ptx::tmem_ld_wait8(t);
#pragma unroll
                  for (int i = 0; i < 8; ++i) t[i] = __float_as_uint(__uint_as_float(t[i]) * a);
                  ptx::tmem_st_32x32b_x8(lane_addr + AQ_O_COL + oc, t);
                }
              }
              if (c > 0) {   // this block's chunk-0 P was taken against the old maximum
                ptx::tmem_st_wait();
#pragma unroll 1
                for (int pc = 0; pc < 16; pc += 8) {
                  uint32_t t[8];
                  ptx::tmem_ld_32x32b_x8(lane_addr + AQ_S_COL + pc, t);
                  ptx::tmem_ld_wait8(t);
#pragma unroll
                  for (int i = 0; i < 8; ++i) {
                    const float lo = ptx::h16_to_f32(F16, static_cast<unsigned short>(t[i] & 0xffffu)) * a;
                    const float hi = ptx::h16_to_f32(F16, static_cast<unsigned short>(t[i] >> 16)) * a;
                    t[i] = ptx::pack_h2<F16>(lo, hi);
                  }
                  ptx::tmem_st_32x32b_x8(lane_addr + AQ_S_COL + pc, t);
                }
              }
              run_exps();
            }
            bsum += csum;
            if constexpr (TL) { if (tl) asm volatile("" ::"f"(csum)); }
            if constexpr (TL) att_stamp(args, tl, 0, j, 3 + 2 * c, p);   // chunk c: exponentials issued
          }
        }
        l_run += bsum;
        ptx::tmem_st_wait();       // P (and a rescaled O) are in TMEM
        ptx::tc_fence_before();    // ... and ordered before the MMA that reads / accumulates on them
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(p_full);
        if constexpr (TL) att_stamp(args, tl, 0, j, 6, p);   // P_j handed to the control thread
      }
      // ---- epilogue: ctx = O / l
      ptx::mbar_wait(o_full, w & 1, 61);
      ptx::tc_fence_after();
      const float inv = 1.0f / l_run;
      uint32_t t[ATT_DH / 32][32];
#pragma unroll
      for (int c = 0; c < ATT_DH / 32; ++c) ptx::tmem_ld_32x32b_x32(lane_addr + AQ_O_COL + c * 32, t[c]);
#pragma unroll
      for (int c = 0; c < ATT_DH / 32; ++c) ptx::tmem_ld_wait(t[c]);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(o_empty);   // the next item's first PV may overwrite O
      int pair, qrow;
      __nv_bfloat16* o;
      bool row_ok;
      if constexpr (VARLEN) {
        int row0, qt, h0, ns;
        att_vdecode(args, it, row0, Ni, qt, h0, ns);
        const int slot_rows = ATT_BQ / ns, sl = r / slot_rows;
        const int h = h0 + sl;
        qrow = qt * ATT_BQ + (r - sl * slot_rows);
        row_ok = h < args.heads && qrow < Ni;   // a ragged tile's rows beyond its image belong to the next image: never written
        o = args.out + static_cast<long long>(row0 + qrow) * args.ldo + h * ATT_DH;
      } else {
      {
        int pair0, qt, ns;
        aq_decode(args, it, pair0, qt, ns);
        const int slot_rows = ATT_BQ / ns, sl = r / slot_rows;   // packed tail item: slot = lane group, one pair each
        pair = pair0 + sl;
        qrow = qt * ATT_BQ + (r - sl * slot_rows);
      }
      row_ok = pair < args.n_pairs && qrow < N;
      if (!row_ok) pair = 0;
      const int b = pair / args.heads, h = pair - b * args.heads;
      o = args.out + static_cast<long long>(b * N + qrow) * args.ldo + h * ATT_DH;
      }
      if (row_ok)
#pragma unroll
      for (int c = 0; c < ATT_DH / 32; ++c) {
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          float v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(t[c][8 * q4 + i]) * inv;
          reinterpret_cast<uint4*>(o + c * 32)[q4] = make_uint4(ptx::pack_h2<F16>(v[0], v[1]), ptx::pack_h2<F16>(v[2], v[3]),
                                                               ptx::pack_h2<F16>(v[4], v[5]), ptx::pack_h2<F16>(v[6], v[7]));
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 4 * AQ_PIPES + 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(ptx::lds_u32(tmem_ptr_smem), 512);
  }
}

}  // namespace vitocm
