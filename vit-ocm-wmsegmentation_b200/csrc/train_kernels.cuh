// Bandwidth-bound kernels of the MIM training step (SSS/mim.py:153-182: loss.backward(), clip_grad_norm_, AdamW):
//   ln_bwd_kernel                        nn.LayerNorm backward (vit.py:107,111,215) fused with the residual-gradient
//                                        accumulation of Block.forward (vit.py:110-111) and the bf16 copy the next GEMMs read
//   attn_delta_kernel                    Delta[q] = sum_d dO[q, d] O[q, d] (flash-attention backward preprocess)
//   dq_convert_kernel                    fp32 dQ accumulator -> bf16 q columns of dQKV (and re-zero the accumulator)
//   mim_loss_bwd_kernel                  model.py:73-76 backward through the masked L1 and PixelShuffle
//   patch_grad_rows_kernel, im2col_bf16_kernel, token_grad_kernel   model.py:29-41 backward (mask-token mix, cls, pos)
//   sumsq_kernel, adamw_kernel           torch.nn.utils.clip_grad_norm_ + torch.optim.AdamW (optimizer.py:73-75)
//   repack_weights_kernel                fp32 masters -> bf16 [R][C] and [C][R] (forward / input-gradient B operands), one launch
// All vectorised and coalesced; statistics and accumulations in fp32 (fp64 for the global gradient norm).
// The backward kernels take the 16-bit element type as a template parameter F16 (false: bf16, true: IEEE fp16).  On fp16
// engines every 16-bit gradient tensor, the fp32 residual gradient dX, dQacc and Delta carry the loss scale S = 2^e chosen by
// mim_loss_bwd_kernel (lscale[0] = S, lscale[1] = 1 / S); the writers of parameter gradients multiply by 1 / S, which is exact.
#pragma once
#include "gemm_sm100.cuh"
#include "ptx.cuh"
#include "vit_kernels.cuh"

namespace vitocm {

__device__ __forceinline__ float bf16lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
// low / high element of a pair of 16-bit values in the format F16 selects
template <bool F16>
__device__ __forceinline__ float h16lo(uint32_t v) {
  if (F16) return __half2float(__ushort_as_half(static_cast<unsigned short>(v & 0xffffu)));
  return bf16lo(v);
}
template <bool F16>
__device__ __forceinline__ float h16hi(uint32_t v) {
  if (F16) return __half2float(__ushort_as_half(static_cast<unsigned short>(v >> 16)));
  return bf16hi(v);
}

// Loss scale of fp16 engines: S = 2^e with |coef| * S in [2^LOSS_SCALE_K0, 2^(LOSS_SCALE_K0 + 1)), coef the loss gradient's
// magnitude (mim_loss_bwd_kernel).  Derived from coef's exponent alone, so a power-of-two change of coef (gscale) changes S
// and nothing else: every scaled 16-bit tensor keeps its bits.  The value of K0 and the headroom it leaves: DESIGN.md §6.
constexpr int LOSS_SCALE_K0 = 0;

// exponent e of the loss scale S = 2^e for a gradient of magnitude a: a S in [2^LOSS_SCALE_K0, 2^(LOSS_SCALE_K0 + 1)); 0 (S = 1)
// when a is 0 or not finite
__device__ __forceinline__ int loss_scale_exp(float a) {
  int e = 0;
  if (a != 0.f && isfinite(a)) {
    int ex;
    frexpf(a, &ex);                          // |a| = f 2^ex, f in [0.5, 1)
    e = LOSS_SCALE_K0 + 1 - ex;
    e = e < -126 ? -126 : (e > 126 ? 126 : e);
  }
  return e;
}

// ------------------------------------------------------------------------------------------------ LayerNorm backward
// One warp per row (grid-stride).  y = (x - mean) * rstd * gamma + beta,  dy = dL/dy (bf16):
//   g = dy * gamma;  dx = rstd * (g - mean(g) - xhat * mean(g * xhat))
//   dX[row] = (accumulate ? dX[row] : 0) + dx   (the residual branch, vit.py:110-111)   and   dXb = bf16(dX)
//   dgamma += dy * xhat,  dbeta += dy           (per-lane partials -> shared memory -> one atomicAdd per block and column)
//   dbias_out += column sums of the new dX      (= the bias gradient of the Linear whose output was added into this
//                                                residual stream: proj of this block / fc2 of the previous one)
// F16: dy / dXb are fp16 and carry the loss scale; dgamma, dbeta and dbias_out are multiplied by lscale[1] = 1 / S.
// SCALED (stochastic depth): dXb and the dbias_out sums use row_scale[row / rows_per_scale] * dX, the gradient that enters the residual
// branch whose output was added into this stream; dX itself (the identity path), dgamma and dbeta are unscaled.
template <int NV, bool F16 = false, bool SCALED = false>
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dy, long long ld_dy, const float* __restrict__ gamma,
              float* __restrict__ dX, __nv_bfloat16* __restrict__ dXb, float* __restrict__ dgamma, float* __restrict__ dbeta,
              float* __restrict__ dbias_out, int accumulate, int M, int D, float eps, const float* __restrict__ lscale = nullptr,
              const float* __restrict__ row_scale = nullptr, int rows_per_scale = 1) {
  constexpr int CNT = NV > 0 ? NV : LN_MAX_VEC;
  extern __shared__ float ln_red[];   // [3][D]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int nvec = D >> 2;
  for (int i = threadIdx.x; i < 3 * D; i += blockDim.x) ln_red[i] = 0.f;
  __syncthreads();
  float4 gm[CNT], accg[CNT], accb[CNT], acco[CNT];
#pragma unroll
  for (int i = 0; i < CNT; ++i) {
    const int idx = lane + 32 * i;
    accg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    accb[i] = accg[i];
    acco[i] = accg[i];
    gm[i] = (NV > 0 || idx < nvec) ? __ldg(reinterpret_cast<const float4*>(gamma) + idx) : accg[i];
  }
  const float inv_d = 1.0f / static_cast<float>(D);
  for (int row = blockIdx.x * nwarps + warp; row < M; row += gridDim.x * nwarps) {
    const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(row) * D);
    const uint2* dr = reinterpret_cast<const uint2*>(dy + static_cast<long long>(row) * ld_dy);
    float4 v[CNT], g[CNT], acc_in[CNT];
    float4* dxr = reinterpret_cast<float4*>(dX + static_cast<long long>(row) * D);
    const float rs = SCALED ? __ldg(row_scale + row / rows_per_scale) : 1.f;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < CNT; ++i) {
      const int idx = lane + 32 * i;
      if (NV > 0 || idx < nvec) {
        v[i] = xr[idx];
        // the running residual gradient is requested together with x and dy: one exposed memory latency per row, not two
        acc_in[i] = accumulate ? dxr[idx] : make_float4(0.f, 0.f, 0.f, 0.f);
        const uint2 d2 = dr[idx];
        g[i] = make_float4(h16lo<F16>(d2.x), h16hi<F16>(d2.x), h16lo<F16>(d2.y), h16hi<F16>(d2.y));
        s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      }
    }
    const float mean = warp_sum(s) * inv_d;
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < CNT; ++i) {
      const int idx = lane + 32 * i;
      if (NV > 0 || idx < nvec) {
        v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
        ss += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
      }
    }
    const float rstd = rsqrtf(warp_sum(ss) * inv_d + eps);
    float c1 = 0.f, c2 = 0.f;
#pragma unroll
    for (int i = 0; i < CNT; ++i) {
      const int idx = lane + 32 * i;
      if (NV > 0 || idx < nvec) {
        v[i].x *= rstd; v[i].y *= rstd; v[i].z *= rstd; v[i].w *= rstd;   // xhat
        accb[i].x += g[i].x; accb[i].y += g[i].y; accb[i].z += g[i].z; accb[i].w += g[i].w;
        accg[i].x += g[i].x * v[i].x; accg[i].y += g[i].y * v[i].y; accg[i].z += g[i].z * v[i].z; accg[i].w += g[i].w * v[i].w;
        g[i].x *= gm[i].x; g[i].y *= gm[i].y; g[i].z *= gm[i].z; g[i].w *= gm[i].w;
        c1 += (g[i].x + g[i].y) + (g[i].z + g[i].w);
        c2 += (g[i].x * v[i].x + g[i].y * v[i].y) + (g[i].z * v[i].z + g[i].w * v[i].w);
      }
    }
    c1 = warp_sum(c1) * inv_d;
    c2 = warp_sum(c2) * inv_d;
    uint2* dbr = reinterpret_cast<uint2*>(dXb + static_cast<long long>(row) * D);
#pragma unroll
    for (int i = 0; i < CNT; ++i) {
      const int idx = lane + 32 * i;
      if (NV > 0 || idx < nvec) {
        float4 o = acc_in[i];
        o.x += rstd * (g[i].x - c1 - v[i].x * c2);
        o.y += rstd * (g[i].y - c1 - v[i].y * c2);
        o.z += rstd * (g[i].z - c1 - v[i].z * c2);
        o.w += rstd * (g[i].w - c1 - v[i].w * c2);
        dxr[idx] = o;
        if (SCALED) { o.x *= rs; o.y *= rs; o.z *= rs; o.w *= rs; }
        dbr[idx] = make_uint2(ptx::pack_h2<F16>(o.x, o.y), ptx::pack_h2<F16>(o.z, o.w));
        acco[i].x += o.x; acco[i].y += o.y; acco[i].z += o.z; acco[i].w += o.w;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < CNT; ++i) {
    const int idx = lane + 32 * i;
    if (NV > 0 || idx < nvec) {
      atomicAdd(ln_red + 4 * idx, accg[i].x); atomicAdd(ln_red + 4 * idx + 1, accg[i].y);
      atomicAdd(ln_red + 4 * idx + 2, accg[i].z); atomicAdd(ln_red + 4 * idx + 3, accg[i].w);
      atomicAdd(ln_red + D + 4 * idx, accb[i].x); atomicAdd(ln_red + D + 4 * idx + 1, accb[i].y);
      atomicAdd(ln_red + D + 4 * idx + 2, accb[i].z); atomicAdd(ln_red + D + 4 * idx + 3, accb[i].w);
      if (dbias_out != nullptr) {
        atomicAdd(ln_red + 2 * D + 4 * idx, acco[i].x); atomicAdd(ln_red + 2 * D + 4 * idx + 1, acco[i].y);
        atomicAdd(ln_red + 2 * D + 4 * idx + 2, acco[i].z); atomicAdd(ln_red + 2 * D + 4 * idx + 3, acco[i].w);
      }
    }
  }
  __syncthreads();
  if (F16) {
    const float inv = lscale != nullptr ? lscale[1] : 1.0f;
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
      atomicAdd(dgamma + i, ln_red[i] * inv);
      atomicAdd(dbeta + i, ln_red[D + i] * inv);
      if (dbias_out != nullptr) atomicAdd(dbias_out + i, ln_red[2 * D + i] * inv);
    }
    return;
  }
  for (int i = threadIdx.x; i < D; i += blockDim.x) {
    atomicAdd(dgamma + i, ln_red[i]);
    atomicAdd(dbeta + i, ln_red[D + i]);
    if (dbias_out != nullptr) atomicAdd(dbias_out + i, ln_red[2 * D + i]);
  }
}

// ------------------------------------------------------------------------------------------------ attention backward helpers
// delta[b][h][q] (row pitch npad) = sum_d dO[row][h*DH + d] * O[row][h*DH + d]; one warp per token row, DH / 32 16-bit values per
// lane per head; all heads' loads are issued before the first reduction (HG heads at a time) so that a row costs one memory latency
template <int HG, int DH = 64, bool F16 = false>
__global__ void __launch_bounds__(256)
attn_delta_kernel(const __nv_bfloat16* __restrict__ O, const __nv_bfloat16* __restrict__ dO, long long ld, float* __restrict__ delta,
                  int B, int N, int heads, int npad) {
  const int lane = threadIdx.x & 31;
  const long long M = static_cast<long long>(B) * N;
  for (long long row = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5); row < M;
       row += static_cast<long long>(gridDim.x) * (blockDim.x >> 5)) {
    const int b = static_cast<int>(row / N), q = static_cast<int>(row - static_cast<long long>(b) * N);
    for (int h0 = 0; h0 < heads; h0 += HG) {
      constexpr int W = DH / 64;   // 32-bit words (bf16 pairs) per lane and head
      uint32_t o[HG][W], d[HG][W];
#pragma unroll
      for (int k = 0; k < HG; ++k) {
        if (h0 + k < heads) {
#pragma unroll
          for (int u = 0; u < W; ++u) {
            o[k][u] = *reinterpret_cast<const uint32_t*>(O + row * ld + (h0 + k) * DH + 2 * (W * lane + u));
            d[k][u] = *reinterpret_cast<const uint32_t*>(dO + row * ld + (h0 + k) * DH + 2 * (W * lane + u));
          }
        }
      }
#pragma unroll
      for (int k = 0; k < HG; ++k) {
        if (h0 + k < heads) {
          float p = h16lo<F16>(o[k][0]) * h16lo<F16>(d[k][0]) + h16hi<F16>(o[k][0]) * h16hi<F16>(d[k][0]);
#pragma unroll
          for (int u = 1; u < W; ++u) p += h16lo<F16>(o[k][u]) * h16lo<F16>(d[k][u]) + h16hi<F16>(o[k][u]) * h16hi<F16>(d[k][u]);
          const float s = warp_sum(p);
          if (lane == 0) delta[(static_cast<long long>(b) * heads + h0 + k) * npad + q] = s;
        }
      }
    }
  }
}

// dqkv[row][0:D] = 16-bit(acc[row][:]);  acc <- 0.  One warp per pair of rows (grid-strided); all loads of a pass (up to
// 2 rows x 4 float4 per lane) are issued before the first store so that a warp keeps 4 KB in flight.
template <bool F16 = false>
__global__ void __launch_bounds__(256)
dq_convert_kernel(float4* __restrict__ acc, __nv_bfloat16* __restrict__ dqkv, long long ld, int M, int D) {
  const int nvec = D >> 2;
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  for (int row0 = 2 * (blockIdx.x * wpb + (threadIdx.x >> 5)); row0 < M; row0 += 2 * gridDim.x * wpb) {
    for (int base = 0; base < nvec; base += 128) {
      float4 v[2][4];
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = base + lane + 32 * u;
          if (row0 + r < M && c < nvec) v[r][u] = acc[static_cast<long long>(row0 + r) * nvec + c];
        }
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int c = base + lane + 32 * u;
          if (row0 + r < M && c < nvec) {
            acc[static_cast<long long>(row0 + r) * nvec + c] = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<uint2*>(dqkv + static_cast<long long>(row0 + r) * ld + 4 * c) =
                make_uint2(ptx::pack_h2<F16>(v[r][u].x, v[r][u].y), ptx::pack_h2<F16>(v[r][u].z, v[r][u].w));
          }
        }
    }
  }
}

// ------------------------------------------------------------------------------------------------ loss backward
// loss = sum |x - x_rec| * mask / (sum mask + 1e-5) / C  (model.py:75-76), x_rec = PixelShuffle(Y) (model.py:61-66):
//   dY[b*(n+1) + 1 + tok][c p^2 + i p + j] = *gscale * mask[b, tok] * sign(x_rec - x) / ((sums[1] + 1e-5) * C)
// CLS rows of dY are zero.  One thread per 8 consecutive columns (one patch row of one channel when p == 8).
// F16: dY is fp16 and multiplied by the loss scale S = 2^e (|coef| S in [2^LOSS_SCALE_K0, 2^(LOSS_SCALE_K0 + 1)); S = 1 when coef
// is 0 or not finite), chosen here on the device from coef's exponent; S and 1 / S go to lscale[0], lscale[1].
template <bool F16 = false>
__global__ void __launch_bounds__(256)
mim_loss_bwd_kernel(const float* __restrict__ x, const float* __restrict__ x_rec, const float* __restrict__ mask,
                    const double* __restrict__ sums, const float* __restrict__ gscale, __nv_bfloat16* __restrict__ dY, int B, int C, int H,
                    int W, int p, float* __restrict__ lscale = nullptr) {
  const int Wp = W / p, n = (H / p) * Wp, ldy = C * p * p, groups = ldy / 8;
  float coef = (gscale != nullptr ? *gscale : 1.0f) / (static_cast<float>(sums[1] + 1e-5) * static_cast<float>(C));
  if (F16) {
    const int e = loss_scale_exp(coef);
    const float S = __int_as_float((127 + e) << 23), inv = __int_as_float((127 - e) << 23);
    coef *= S;                               // exact
    if (blockIdx.x == 0 && threadIdx.x == 0 && lscale != nullptr) {
      lscale[0] = S;
      lscale[1] = inv;
    }
  }
  const long long total = static_cast<long long>(B) * (n + 1) * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long row = idx / groups;
    const int col = static_cast<int>(idx - row * groups) * 8;
    const int b = static_cast<int>(row / (n + 1)), t = static_cast<int>(row - static_cast<long long>(b) * (n + 1));
    float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (t > 0) {
      const int tok = t - 1, py = tok / Wp, px = tok - py * Wp;
      const float m = mask[static_cast<long long>(b) * n + tok] * coef;
      if (m != 0.f) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int cc = col + k;
          const int c = cc / (p * p), rem = cc - c * p * p, i = rem / p, j = rem - i * p;
          const long long pix = ((static_cast<long long>(b) * C + c) * H + py * p + i) * W + px * p + j;
          const float d = x_rec[pix] - x[pix];
          g[k] = d > 0.f ? m : (d < 0.f ? -m : 0.f);
        }
      }
    }
    *reinterpret_cast<uint4*>(dY + row * ldy + col) =
        make_uint4(ptx::pack_h2<F16>(g[0], g[1]), ptx::pack_h2<F16>(g[2], g[3]), ptx::pack_h2<F16>(g[4], g[5]), ptx::pack_h2<F16>(g[6], g[7]));
  }
}

// ------------------------------------------------------------------------------------------------ encoder gradient seeding
// vitocm_encoder_backward: the caller's upstream gradient dfeats (fp32) becomes the 16-bit dy of the final norm's backward.
// amax_bits[0] = max |g| as float bits (non-negative floats order like their bit patterns; NaN orders above +inf).  Zeroed by
// the caller.
__global__ void __launch_bounds__(256)
grad_amax_kernel(const float4* __restrict__ g, long long n4, unsigned* __restrict__ amax_bits) {
  unsigned m = 0u;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = g[i];
    m = max(m, max(max(__float_as_uint(v.x) & 0x7fffffffu, __float_as_uint(v.y) & 0x7fffffffu),
                   max(__float_as_uint(v.z) & 0x7fffffffu, __float_as_uint(v.w) & 0x7fffffffu)));
  }
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(amax_bits, m);
}

// out[i] = 16-bit(g[i] * S).  F16: S = 2^loss_scale_exp(amax) from grad_amax_kernel's result (S = 1 for an all-zero or non-finite
// gradient), written with 1 / S to lscale[0], lscale[1] as mim_loss_bwd_kernel does; a power-of-two change of g changes S and
// nothing else.  bf16: S = 1, nothing read or written besides g and out.
template <bool F16 = false>
__global__ void __launch_bounds__(256)
seed_grad_kernel(const float4* __restrict__ g, long long n4, const unsigned* __restrict__ amax_bits, __nv_bfloat16* __restrict__ out,
                 float* __restrict__ lscale) {
  float S = 1.0f;
  if (F16) {
    const int e = loss_scale_exp(__uint_as_float(*amax_bits));
    S = __int_as_float((127 + e) << 23);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      lscale[0] = S;
      lscale[1] = __int_as_float((127 - e) << 23);
    }
  }
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = g[i];
    *reinterpret_cast<uint2*>(out + 4 * i) = make_uint2(ptx::pack_h2<F16>(v.x * S, v.y * S), ptx::pack_h2<F16>(v.z * S, v.w * S));
  }
}

// ------------------------------------------------------------------------------------------------ token-embedding backward
// G[b*n + i][:] = 16-bit((1 - mask[b, i]) * dX0[b, 1 + i, :])    (model.py:31-33: only unmasked patches see the conv; mask NULL: 0)
template <bool F16 = false>
__global__ void __launch_bounds__(256)
patch_grad_rows_kernel(const float4* __restrict__ dX0, const float* __restrict__ mask, __nv_bfloat16* __restrict__ G, int B, int n, int D) {
  const int nvec = D >> 2;
  const long long total = static_cast<long long>(B) * n * nvec;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = idx / nvec;
    const int c = static_cast<int>(idx - m * nvec);
    const int b = static_cast<int>(m / n), i = static_cast<int>(m - static_cast<long long>(b) * n);
    const float w = mask != nullptr ? 1.0f - mask[m] : 1.0f;
    const float4 v = dX0[(static_cast<long long>(b) * (n + 1) + 1 + i) * nvec + c];
    *reinterpret_cast<uint2*>(G + m * D + 4 * c) = make_uint2(ptx::pack_h2<F16>(v.x * w, v.y * w), ptx::pack_h2<F16>(v.z * w, v.w * w));
  }
}

// P[b*n + py*Wp + px][c p^2 + yi p + xi] = 16-bit(x[b, c, py p + yi, px p + xi]); one thread per 8 consecutive pixels
template <bool F16 = false>
__global__ void __launch_bounds__(256)
im2col_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ P, int B, int C, int H, int W, int p) {
  const int Wp = W / p, n = (H / p) * Wp, K = C * p * p, groups = K / 8;
  const long long total = static_cast<long long>(B) * n * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = idx / groups;
    const int k = static_cast<int>(idx - m * groups) * 8;
    const int b = static_cast<int>(m / n), i = static_cast<int>(m - static_cast<long long>(b) * n);
    const int py = i / Wp, px = i - py * Wp;
    const int c = k / (p * p), rem = k - c * p * p, yi = rem / p, xi = rem - yi * p;
    const float* src = x + ((static_cast<long long>(b) * C + c) * H + py * p + yi) * W + px * p + xi;
    const float4 a = *reinterpret_cast<const float4*>(src), bq = *reinterpret_cast<const float4*>(src + 4);
    *reinterpret_cast<uint4*>(P + m * K + k) =
        make_uint4(ptx::pack_h2<F16>(a.x, a.y), ptx::pack_h2<F16>(a.z, a.w), ptx::pack_h2<F16>(bq.x, bq.y), ptx::pack_h2<F16>(bq.z, bq.w));
  }
}

// inverse of im2col_bf16_kernel for the input gradient: dx[b, c, py p + yi, px p + xi] = dP[b*n + py*Wp + px][c p^2 + yi p + xi] *
// (*inv_scale, NULL: 1).  Patches do not overlap, so every pixel has exactly one source: a permutation, no atomics.
__global__ void __launch_bounds__(256)
col2im_dx_kernel(const float* __restrict__ dP, float* __restrict__ dx, int B, int C, int H, int W, int p, const float* __restrict__ inv_scale) {
  const int Wp = W / p, n = (H / p) * Wp, K = C * p * p, groups = K / 8;
  const float s = inv_scale != nullptr ? *inv_scale : 1.0f;
  const long long total = static_cast<long long>(B) * n * groups;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long m = idx / groups;
    const int k = static_cast<int>(idx - m * groups) * 8;
    const int b = static_cast<int>(m / n), i = static_cast<int>(m - static_cast<long long>(b) * n);
    const int py = i / Wp, px = i - py * Wp;
    const int c = k / (p * p), rem = k - c * p * p, yi = rem / p, xi = rem - yi * p;
    const float4 a = *reinterpret_cast<const float4*>(dP + m * K + k), bq = *reinterpret_cast<const float4*>(dP + m * K + k + 4);
    float* dst = dx + ((static_cast<long long>(b) * C + c) * H + py * p + yi) * W + px * p + xi;
    *reinterpret_cast<float4*>(dst) = make_float4(a.x * s, a.y * s, a.z * s, a.w * s);
    *reinterpret_cast<float4*>(dst + 4) = make_float4(bq.x * s, bq.y * s, bq.z * s, bq.w * s);
  }
}

// dpos[t][:] = sum_b dX0[b, t, :];  dcls += dpos[0];  dmask_token += sum_{b, i} mask[b, i] * dX0[b, 1 + i, :]  (mask NULL: no mix)
// one thread per (token t, float4 column group), looping over the batch.  F16: dX0 carries the loss scale; the sums are
// multiplied by lscale[1] = 1 / S
template <bool F16 = false>
__global__ void __launch_bounds__(256)
token_grad_kernel(const float4* __restrict__ dX0, const float* __restrict__ mask, float4* __restrict__ dpos, float* __restrict__ dcls,
                  float* __restrict__ dmask_token, int B, int n, int D, const float* __restrict__ lscale = nullptr) {
  const int nvec = D >> 2;
  const int total = (n + 1) * nvec;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int t = idx / nvec, c = idx - t * nvec;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), sm = s;
  for (int b = 0; b < B; ++b) {
    const float4 v = dX0[(static_cast<long long>(b) * (n + 1) + t) * nvec + c];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    if (t > 0 && mask != nullptr) {
      const float w = mask[static_cast<long long>(b) * n + t - 1];
      sm.x += w * v.x; sm.y += w * v.y; sm.z += w * v.z; sm.w += w * v.w;
    }
  }
  if (F16) {
    const float inv = lscale != nullptr ? lscale[1] : 1.0f;
    s.x *= inv; s.y *= inv; s.z *= inv; s.w *= inv;
    sm.x *= inv; sm.y *= inv; sm.z *= inv; sm.w *= inv;
  }
  dpos[idx] = s;
  if (t == 0) {
    atomicAdd(dcls + 4 * c, s.x); atomicAdd(dcls + 4 * c + 1, s.y); atomicAdd(dcls + 4 * c + 2, s.z); atomicAdd(dcls + 4 * c + 3, s.w);
  } else if (dmask_token != nullptr) {
    atomicAdd(dmask_token + 4 * c, sm.x); atomicAdd(dmask_token + 4 * c + 1, sm.y);
    atomicAdd(dmask_token + 4 * c + 2, sm.z); atomicAdd(dmask_token + 4 * c + 3, sm.w);
  }
}

// ------------------------------------------------------------------------------------------------ optimizer
// out[0] += sum g^2 (fp64): the squared global gradient norm of torch.nn.utils.clip_grad_norm_ (mim.py:176)
__global__ void __launch_bounds__(256)
sumsq_kernel(const float4* __restrict__ g, long long n4, const float* __restrict__ tail, int ntail, double* __restrict__ out) {
  __shared__ double red[8];
  double s = 0.0;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float4 v = g[i];
    s += static_cast<double>(v.x * v.x + v.y * v.y) + static_cast<double>(v.z * v.z + v.w * v.w);
  }
  if (blockIdx.x == 0 && static_cast<int>(threadIdx.x) < ntail) s += static_cast<double>(tail[threadIdx.x]) * tail[threadIdx.x];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (blockDim.x >> 5); ++w) t += red[w];
    atomicAdd(out, t);
  }
}

// second half of clip_grad_norm_ applied in place: g <- g * min(1, max_norm / (sqrt(sumsq) + 1e-6)); the coefficient is formed on
// the device from the sum of squares (no host sync)
__global__ void __launch_bounds__(256)
grad_clip_kernel(float4* __restrict__ g, long long n4, float* __restrict__ tail, int ntail, const double* __restrict__ sumsq, float max_norm) {
  const float c = max_norm / (static_cast<float>(sqrt(*sumsq)) + 1e-6f);
  if (!(c < 1.0f)) return;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float4 v = g[i];
    v.x *= c; v.y *= c; v.z *= c; v.w *= c;
    g[i] = v;
  }
  if (blockIdx.x == 0 && static_cast<int>(threadIdx.x) < ntail) tail[threadIdx.x] *= c;
}

struct AdamWArgs {
  float lr, beta1, beta2, eps, weight_decay;
  float bias_corr1, bias_corr2_sqrt;   // 1 - beta1^t, sqrt(1 - beta2^t)
  float max_norm;                      // <= 0: no clipping
  float grad_scale;                    // applied to the gradient before everything else (e.g. 1 / world size)
};

// torch.optim.AdamW (decoupled weight decay) with the clip coefficient of clip_grad_norm_ folded in:
//   coef = min(1, max_norm / (sqrt(sumsq) * grad_scale + 1e-6));  g <- g * grad_scale * coef   (also written back)
//   p <- p * (1 - lr * wd);  m <- b1 m + (1 - b1) g;  v <- b2 v + (1 - b2) g^2
//   p <- p - (lr / bc1) * m / (sqrt(v) / sqrt(bc2) + eps)
// decay[i] != 0 selects weight decay per element (1-D parameters and biases have none, optimizer.py:14-33).
__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
             const uint8_t* __restrict__ decay, long long n, const double* __restrict__ sumsq, AdamWArgs a) {
  float coef = a.grad_scale;
  if (a.max_norm > 0.f && sumsq != nullptr) {
    const float total = static_cast<float>(sqrt(*sumsq)) * a.grad_scale;
    const float c = a.max_norm / (total + 1e-6f);
    coef *= c < 1.0f ? c : 1.0f;
  }
  const float step = a.lr / a.bias_corr1;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * coef;
    float pi = p[i];
    if (decay[i]) pi *= 1.0f - a.lr * a.weight_decay;
    const float mi = a.beta1 * m[i] + (1.0f - a.beta1) * gi;
    const float vi = a.beta2 * v[i] + (1.0f - a.beta2) * gi * gi;
    pi -= step * mi / (sqrtf(vi) / a.bias_corr2_sqrt + a.eps);
    g[i] = gi;
    p[i] = pi;
    m[i] = mi;
    v[i] = vi;
  }
}

// One launch for every Linear weight of the model (bf16 engines): fp32 master [R][C] -> bf16 [R][C] (forward B operand) and
// bf16 [C][R] (input-gradient B operand).  blockIdx.x walks 32 x 32 tiles; the table gives each matrix its first tile.
struct RepackEntry {
  const float* src;
  __nv_bfloat16* dst;     // [R][C] or nullptr
  __nv_bfloat16* dst_t;   // [C][R] or nullptr
  int R, C;
  int tile0;              // index of this matrix's first tile
  int tiles_c;            // tiles per row of tiles
};
__global__ void __launch_bounds__(256)
repack_weights_kernel(const RepackEntry* __restrict__ table, int n_entries, int f16 = 0 /*fp16 engines: IEEE half operands*/) {
  __shared__ float tile[32][33];
  int lo = 0, hi = n_entries - 1;
  const int t = blockIdx.x;
  while (lo < hi) {            // last entry whose tile0 <= t
    const int mid = (lo + hi + 1) >> 1;
    if (table[mid].tile0 <= t) lo = mid; else hi = mid - 1;
  }
  const RepackEntry e = table[lo];
  const int local = t - e.tile0;
  const int r0 = (local / e.tiles_c) * 32, c0 = (local % e.tiles_c) * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int k = ty; k < 32; k += 8) {
    const int r = r0 + k, c = c0 + tx;
    float v = 0.f;
    if (r < e.R && c < e.C) {
      v = e.src[static_cast<long long>(r) * e.C + c];
      if (e.dst != nullptr) {
        if (f16) reinterpret_cast<__half*>(e.dst)[static_cast<long long>(r) * e.C + c] = __float2half_rn(ptx::f16_round(v));
        else e.dst[static_cast<long long>(r) * e.C + c] = __float2bfloat16_rn(v);
      }
    }
    tile[k][tx] = v;
  }
  if (e.dst_t == nullptr) return;
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k, r = r0 + tx;
    if (c < e.C && r < e.R) {
      if (f16) reinterpret_cast<__half*>(e.dst_t)[static_cast<long long>(c) * e.R + r] = __float2half_rn(ptx::f16_round(tile[tx][k]));
      else e.dst_t[static_cast<long long>(c) * e.R + r] = __float2bfloat16_rn(tile[tx][k]);
    }
  }
}

}  // namespace vitocm
