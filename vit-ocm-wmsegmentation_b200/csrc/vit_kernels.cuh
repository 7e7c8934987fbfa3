// Bandwidth-bound ViT kernels (vectorised, coalesced, fp32 statistics):
//   cls_rows_kernel      SSS/dino/vision_transformer.py:203-207, CLS row (patch rows: gemm_sm100.cuh A_PATCH)
//   layernorm_kernel     vit.py:107,111 (norm1/norm2) and :215/:234 (final norm), eps = 1e-6
//   cls_attn_row_kernel  vit.py:80-84 restricted to the CLS query (or a list of query tokens, SSS/analyse_attention.py:183-247) of the last block
//   attn_probs_kernel    vit.py:83-84 full softmax(QK^T) (API-complete get_last_selfattention)
//   mim_shuffle_loss_kernel  SSS/model.py:61-66,73-76 (PixelShuffle + masked L1 of MIM.forward)
#pragma once
#include "ptx.cuh"

namespace vitocm {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------------------
// prepare_tokens, CLS part (vit.py:203-207): X[b, 0, :] = cls_token + pos[0].  The patch rows are
// written by the patch-embedding GEMM (gemm_sm100.cuh, A_PATCH / EPI_PATCH_F32).
// ---------------------------------------------------------------------------------------
__global__ void cls_rows_kernel(const float* __restrict__ cls_token, const float* __restrict__ pos, float* __restrict__ X, int B,
                                long long image_stride, int D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * D) return;
  const int b = i / D, d = i - b * D;
  X[static_cast<long long>(b) * image_stride + d] = cls_token[d] + pos[d];
}
// the same for images of different sizes packed back to back (vimg as GemmArgs::vimg): image b's CLS row is token row vimg[b].x + b,
// its position row pos[vimg[b].z]
__global__ void cls_rows_var_kernel(const float* __restrict__ cls_token, const float* __restrict__ pos, const int4* __restrict__ vimg,
                                    float* __restrict__ X, int B, int D) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * D) return;
  const int b = i / D, d = i - b * D;
  const int4 g = vimg[b];
  X[static_cast<long long>(g.x + b) * D + d] = cls_token[d] + pos[static_cast<long long>(g.z) * D + d];
}

// ---------------------------------------------------------------------------------------
// LayerNorm over the last dim of the fp32 token stream, one warp per row, float4 loads.
// Outputs: bf16 (hi) and, in split mode, lo = bf16(y - hi) at column offset lo_off of the same
// row (the A operand of the following GEMM); optionally the fp32 result (final norm -> feat).
// ---------------------------------------------------------------------------------------
constexpr int LN_MAX_VEC = 8;  // up to D = 8*32*4 = 1024

// NV > 0: D == NV * 128 exactly (no predicates: 3 float4 per lane for ViT-S, 6 for ViT-B); NV == 0: any D % 4 == 0.
template <int NV>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                 __nv_bfloat16* __restrict__ out_bf16, long long ldo, int split, int lo_off,
                 float* __restrict__ out_f32, long long ldf, int M, int D, float eps, float* __restrict__ x_copy = nullptr,
                 int f16 = 0 /*16-bit output format: 0 = bf16, 1 = IEEE fp16*/) {
  constexpr int CNT = NV > 0 ? NV : LN_MAX_VEC;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + static_cast<long long>(row) * D);
  const int nvec = D >> 2;
  float4 v[CNT];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < CNT; ++i) {
    const int idx = lane + 32 * i;
    if (NV > 0 || idx < nvec) {
      v[i] = xr[idx];
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      // training: snapshot of the row this LayerNorm saw (its backward needs x, the residual stream moves on in place)
      if (x_copy != nullptr) reinterpret_cast<float4*>(x_copy + static_cast<long long>(row) * D)[idx] = v[i];
    }
  }
  const float inv_d = 1.0f / static_cast<float>(D);
  const float mean = warp_sum(s) * inv_d;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < CNT; ++i) {
    const int idx = lane + 32 * i;
    if (NV > 0 || idx < nvec) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      ss += (a * a + b * b) + (c * c + d * d);
    }
  }
  const float rstd = rsqrtf(warp_sum(ss) * inv_d + eps);
#pragma unroll
  for (int i = 0; i < CNT; ++i) {
    const int idx = lane + 32 * i;
    if (NV > 0 || idx < nvec) {
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + idx);
      const float4 bb = __ldg(reinterpret_cast<const float4*>(beta) + idx);
      float4 y;
      y.x = (v[i].x - mean) * rstd * g.x + bb.x;
      y.y = (v[i].y - mean) * rstd * g.y + bb.y;
      y.z = (v[i].z - mean) * rstd * g.z + bb.z;
      y.w = (v[i].w - mean) * rstd * g.w + bb.w;
      if (out_bf16 != nullptr) {
        __nv_bfloat16* o = out_bf16 + static_cast<long long>(row) * ldo + idx * 4;
        if (f16) {
          *reinterpret_cast<uint2*>(o) = make_uint2(ptx::pack_f16x2(y.x, y.y), ptx::pack_f16x2(y.z, y.w));
          if (split) {
            *reinterpret_cast<uint2*>(o + lo_off) =
                make_uint2(ptx::pack_f16x2(y.x - ptx::f16_round(y.x), y.y - ptx::f16_round(y.y)),
                           ptx::pack_f16x2(y.z - ptx::f16_round(y.z), y.w - ptx::f16_round(y.w)));
          }
        } else {
          *reinterpret_cast<uint2*>(o) = make_uint2(ptx::pack_bf16x2(y.x, y.y), ptx::pack_bf16x2(y.z, y.w));
          if (split) {
            *reinterpret_cast<uint2*>(o + lo_off) =
                make_uint2(ptx::pack_bf16x2(y.x - ptx::bf16_round(y.x), y.y - ptx::bf16_round(y.y)),
                           ptx::pack_bf16x2(y.z - ptx::bf16_round(y.z), y.w - ptx::bf16_round(y.w)));
          }
        }
      }
      if (out_f32 != nullptr) reinterpret_cast<float4*>(out_f32 + static_cast<long long>(row) * ldf)[idx] = y;
    }
  }
}

// ---------------------------------------------------------------------------------------
// Last block, CLS query only (the slice every hot-path caller reads, SSS/utils.py:232 with
// query = 0): one block per (head, image):
//   xn  = LayerNorm(X[b, 0, :])                       (fp32)
//   q_h = Wq[h*DH:(h+1)*DH, :] . xn + bq              (fp32 weights, fp32 math)
//   out[b, h, j] = softmax_j( scale * q_h . K[b, j, h*DH:(h+1)*DH] )   for j in [0, N)
// K comes from the (split-precision) K-projection GEMM as fp32 [B*N, D].  DH = head_dim (64 or 128).
// VAR: the CLS query of images of different sizes packed back to back; `queries` then carries vimg (int4 [B + 1], as GemmArgs::vimg):
// image b has N_b = vimg[b + 1].x - vimg[b].x + 1 tokens from token row vimg[b].x + b on, its rows are out[heads (vimg[b].x + b) ...]
// as [H][N_b], and N is the largest N_b (it sizes the shared memory).
// ---------------------------------------------------------------------------------------
template <int DH, bool VAR = false>
__global__ void __launch_bounds__(256)
cls_attn_row_kernel(const float* __restrict__ X, const float* __restrict__ ln_w, const float* __restrict__ ln_b, float eps,
                    const float* __restrict__ Wq /*[D][D] rows = q outputs*/, const float* __restrict__ bq,
                    const float* __restrict__ Kmat /*[B*N][D] fp32*/, float* __restrict__ out /*[B][H][nq][N]*/, int N, int D,
                    int heads, float scale, const int* __restrict__ queries /*[nq] token indices or nullptr = {0}*/, int nq) {
  extern __shared__ float cls_smem[];  // xn[D] | q[DH] | logits[N] | red[32]
  float* xn = cls_smem;
  float* qv = xn + D;
  float* logits = qv + DH;
  float* red = logits + N;
  const int h = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int qi = blockIdx.z;
  const int4* vimg = reinterpret_cast<const int4*>(queries);
  const long long vrow0 = VAR ? static_cast<long long>(vimg[b].x) + b : 0;   // VAR: the image's first token row and its tokens
  const int vn = VAR ? vimg[b + 1].x - vimg[b].x + 1 : 0;
  const int token = VAR ? 0 : (queries != nullptr ? queries[qi] : 0);    // 0 = the CLS token (SSS/utils.py:232, query = 0)
  const float* xr = X + ((VAR ? vrow0 : static_cast<long long>(b) * N) + token) * D;

  // LayerNorm of the CLS row (block-wide two-pass)
  float s = 0.f;
  for (int d = tid; d < D; d += blockDim.x) s += xr[d];
  s = warp_sum(s);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  float tot = 0.f;
  for (int w = 0; w < nwarps; ++w) tot += red[w];
  const float mean = tot / static_cast<float>(D);
  __syncthreads();
  float ss = 0.f;
  for (int d = tid; d < D; d += blockDim.x) {
    const float c = xr[d] - mean;
    ss += c * c;
  }
  ss = warp_sum(ss);
  if (lane == 0) red[warp] = ss;
  __syncthreads();
  tot = 0.f;
  for (int w = 0; w < nwarps; ++w) tot += red[w];
  const float rstd = rsqrtf(tot / static_cast<float>(D) + eps);
  for (int d = tid; d < D; d += blockDim.x) xn[d] = (xr[d] - mean) * rstd * ln_w[d] + ln_b[d];
  __syncthreads();

  // q_h: DH outputs, one warp per output (coalesced weight rows)
  for (int o = warp; o < DH; o += nwarps) {
    const float* wr = Wq + static_cast<long long>(h * DH + o) * D;
    float acc = 0.f;
    for (int d = lane; d < D; d += 32) acc = fmaf(wr[d], xn[d], acc);
    acc = warp_sum(acc);
    if (lane == 0) qv[o] = acc + bq[h * DH + o];
  }
  __syncthreads();

  // logits: one warp per key, DH / 32 channels per lane
  float lmax = -INFINITY;
  if constexpr (DH == 64) {
    const float q0 = qv[2 * lane], q1 = qv[2 * lane + 1];
    for (int j = warp; j < (VAR ? vn : N); j += nwarps) {
      const float2 kk = *reinterpret_cast<const float2*>(Kmat + ((VAR ? vrow0 : static_cast<long long>(b) * N) + j) * D + h * 64 + 2 * lane);
      float acc = warp_sum(fmaf(q0, kk.x, q1 * kk.y)) * scale;
      if (lane == 0) logits[j] = acc;
      lmax = fmaxf(lmax, acc);
    }
  } else {
    const float4 qq = reinterpret_cast<const float4*>(qv)[lane];
    for (int j = warp; j < (VAR ? vn : N); j += nwarps) {
      const float4 kk = *reinterpret_cast<const float4*>(Kmat + ((VAR ? vrow0 : static_cast<long long>(b) * N) + j) * D + h * DH + 4 * lane);
      float acc = warp_sum(fmaf(qq.x, kk.x, fmaf(qq.y, kk.y, fmaf(qq.z, kk.z, qq.w * kk.w)))) * scale;
      if (lane == 0) logits[j] = acc;
      lmax = fmaxf(lmax, acc);
    }
  }
  if (lane == 0) red[warp] = lmax;
  __syncthreads();
  float gmax = -INFINITY;
  for (int w = 0; w < nwarps; ++w) gmax = fmaxf(gmax, red[w]);
  __syncthreads();
  float lsum = 0.f;
  for (int j = tid; j < (VAR ? vn : N); j += blockDim.x) {
    const float e = expf(logits[j] - gmax);
    logits[j] = e;
    lsum += e;
  }
  lsum = warp_sum(lsum);
  if (lane == 0) red[warp] = lsum;
  __syncthreads();
  float gsum = 0.f;
  for (int w = 0; w < nwarps; ++w) gsum += red[w];
  const float inv = 1.0f / gsum;
  float* o = VAR ? out + vrow0 * heads + static_cast<long long>(h) * vn : out + ((static_cast<long long>(b) * heads + h) * nq + qi) * N;
  for (int j = tid; j < (VAR ? vn : N); j += blockDim.x) o[j] = logits[j] * inv;
}

// ---------------------------------------------------------------------------------------
// Full attention probabilities of one block, fp32 math on CUDA cores (API-complete path for
// get_last_selfattention / get_intermediate_feat; the hot path never materialises N x N).
// Reads q and k from an fp32 [B*N, 3D] activation.  One block = (qrows-query group, head, image);
// K_h is staged once per block in smem as fp32 with a padded row (DH + 1 floats) so that the
// lane-per-key dot products are bank-conflict free.  DH = head_dim (64 or 128).
// ---------------------------------------------------------------------------------------
constexpr int AP_QROWS = 16;

template <int DH>
__global__ void __launch_bounds__(256)
attn_probs_kernel(const float* __restrict__ qkv /*[B*N][3D]*/, float* __restrict__ attn /*[B][H][N][N]*/, int N, int D,
                  int heads, float scale, int kchunk /*keys staged per pass*/, int qrows) {
  extern __shared__ float ap_smem[];  // K chunk [kchunk][DH + 1] | q [qrows][DH] | logits [qrows][N]
  constexpr int KP = DH + 1;
  float* ks = ap_smem;
  float* qs = ks + kchunk * KP;
  float* lg = qs + qrows * DH;
  const int q0 = blockIdx.x * qrows, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const long long ld = 3LL * D;
  const float* base = qkv + static_cast<long long>(b) * N * ld;
  constexpr int LOG_DH = DH == 64 ? 6 : 7;
  for (int i = tid; i < qrows * DH; i += blockDim.x) {
    const int r = i >> LOG_DH, c = i & (DH - 1);
    qs[i] = (q0 + r < N) ? base[(q0 + r) * ld + h * DH + c] : 0.f;
  }
  for (int k0 = 0; k0 < N; k0 += kchunk) {
    const int kn = min(kchunk, N - k0);
    __syncthreads();
    for (int i = tid; i < kn * DH; i += blockDim.x) {
      const int r = i >> LOG_DH, c = i & (DH - 1);
      ks[r * KP + c] = base[(k0 + r) * ld + D + h * DH + c];
    }
    __syncthreads();
    // each warp: 2 query rows; lane-per-key
    for (int r = warp; r < qrows; r += nwarps) {
      const float* qr = qs + r * DH;
      for (int j = lane; j < kn; j += 32) {
        const float* kr = ks + j * KP;
        float acc = 0.f;
#pragma unroll 16
        for (int c = 0; c < DH; ++c) acc = fmaf(qr[c], kr[c], acc);
        lg[r * N + k0 + j] = acc * scale;
      }
    }
  }
  __syncthreads();
  for (int r = warp; r < qrows; r += nwarps) {
    if (q0 + r >= N) continue;
    float* lr = lg + r * N;
    float mx = -INFINITY;
    for (int j = lane; j < N; j += 32) mx = fmaxf(mx, lr[j]);
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < N; j += 32) {
      const float e = expf(lr[j] - mx);
      lr[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    float* o = attn + ((static_cast<long long>(b) * heads + h) * N + (q0 + r)) * N;
    for (int j = lane; j < N; j += 32) o[j] = lr[j] * inv;
  }
}

// ---------------------------------------------------------------------------------------
// MIM.forward tail (SSS/model.py:61-66, :73-76): PixelShuffle(p) of the 1x1-conv decoder output and the
// masked L1 reconstruction loss.  Y [B][1 + n][C*p*p] fp32 is the decoder GEMM over the normed tokens
// (row 0 of each image = CLS, ignored); x [B][C][H][W]; mask [B][n] in {0,1}.
//   x_rec[b, c, py*p + i, px*p + j] = Y[b, 1 + py*Wp + px, c*p*p + i*p + j]
//   sums[0] += sum |x - x_rec| * mask(py, px)   (over all channels),   sums[1] += sum mask (per pixel)
// loss = sums[0] / (sums[1] + 1e-5) / C is formed by the caller (two doubles, accumulated with atomics).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
mim_shuffle_loss_kernel(const float* __restrict__ Y, const float* __restrict__ x, const float* __restrict__ mask,
                        float* __restrict__ x_rec, double* __restrict__ sums, int B, int C, int H, int W, int p) {
  __shared__ double red[2][8];
  const int Wp = W / p, n = (H / p) * Wp, ldy = C * p * p;
  const long long total = static_cast<long long>(B) * C * H * W;
  double s_abs = 0.0, s_msk = 0.0;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int xx = static_cast<int>(idx % W);
    const int yy = static_cast<int>((idx / W) % H);
    const int c = static_cast<int>((idx / (static_cast<long long>(W) * H)) % C);
    const int b = static_cast<int>(idx / (static_cast<long long>(W) * H * C));
    const int py = yy / p, i = yy - py * p, px = xx / p, j = xx - px * p;
    const int tok = py * Wp + px;
    const float r = Y[(static_cast<long long>(b) * (n + 1) + 1 + tok) * ldy + c * p * p + i * p + j];
    x_rec[idx] = r;
    const float m = mask[static_cast<long long>(b) * n + tok];
    s_abs += static_cast<double>(fabsf(x[idx] - r) * m);
    if (c == 0) s_msk += static_cast<double>(m);
  }
  for (int o = 16; o > 0; o >>= 1) {
    s_abs += __shfl_xor_sync(0xffffffffu, s_abs, o);
    s_msk += __shfl_xor_sync(0xffffffffu, s_msk, o);
  }
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s_abs; red[1][threadIdx.x >> 5] = s_msk; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, m = 0.0;
    for (int w = 0; w < (blockDim.x >> 5); ++w) { a += red[0][w]; m += red[1][w]; }
    atomicAdd(sums, a);
    atomicAdd(sums + 1, m);
  }
}

// bf16 (hi [+ lo]) activation -> fp32 (qkv / ctx export for the API-complete path)
__global__ void bf16_to_f32_kernel(const __nv_bfloat16* __restrict__ in, long long ldi, int split, int lo_off,
                                   float* __restrict__ out, long long ldo, int M, int ncols, int f16 = 0) {
  const unsigned short* in16 = reinterpret_cast<const unsigned short*>(in);
  const long long total = static_cast<long long>(M) * ncols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / ncols;
    const int c = static_cast<int>(i - r * ncols);
    float v = ptx::h16_to_f32(f16 != 0, in16[r * ldi + c]);
    if (split) v += ptx::h16_to_f32(f16 != 0, in16[r * ldi + lo_off + c]);
    out[r * ldo + c] = v;
  }
}

// Patch filter folded over the input channels: out[d][k] = sum_c w[d][c][k] (k over the p*p taps).  A gray image fed as
// R = G = B (every OCM tile of the reference, SURVEY.md 8a F1) then needs K = p*p instead of C*p*p in the patch-embedding GEMM.
__global__ void fold_patch_weight_kernel(const float* __restrict__ w, float* __restrict__ out, int D, int C, int pp) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D * pp) return;
  const int d = i / pp, k = i - d * pp;
  float s = 0.f;
  for (int c = 0; c < C; ++c) s += w[(static_cast<long long>(d) * C + c) * pp + k];
  out[i] = s;
}

// fp32 [R, C] weight -> bf16 hi (and lo) [R, ldo]  (weight repack at load time)
__global__ void split_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, long long ldo, int split,
                                    int lo_off, int R, int C, int f16 = 0) {
  const long long total = static_cast<long long>(R) * C;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / C;
    const int c = static_cast<int>(i - r * C);
    const float v = w[i];
    if (f16) {
      __half* oh = reinterpret_cast<__half*>(out);
      const float hi = ptx::f16_round(v);
      oh[r * ldo + c] = __float2half_rn(hi);
      if (split) oh[r * ldo + lo_off + c] = __float2half_rn(ptx::f16_round(v - hi));
    } else {
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      out[r * ldo + c] = hi;
      if (split) out[r * ldo + lo_off + c] = __float2bfloat16_rn(v - __bfloat162float(hi));
    }
  }
}

// LayerNorm affine parameters folded into the Linear that reads the normalised rows (block_tail_sm100.cuh, TailArgs::fold2 / foldn):
//   W'[n][k] = W[n][k] gamma[k]  (16-bit, K-major, the engine's operand format),   b'[n] = b[n] + sum_k W[n][k] beta[k]  (fp32)
// so that  (xhat gamma + beta) . W^T + b  ==  xhat . W'^T + b'  with xhat = (x - mean) rstd.  One warp per output row.
__global__ void fold_ln_weight_kernel(const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, __nv_bfloat16* __restrict__ out, float* __restrict__ bias_out,
                                      int R, int C, int f16) {
  const int row = static_cast<int>((blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= R) return;
  const float* wr = w + static_cast<long long>(row) * C;
  float acc = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float v = wr[c];
    acc = fmaf(v, beta[c], acc);
    const float s = v * gamma[c];
    if (f16) reinterpret_cast<__half*>(out)[static_cast<long long>(row) * C + c] = __float2half_rn(s);
    else out[static_cast<long long>(row) * C + c] = __float2bfloat16_rn(s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) bias_out[row] = bias[row] + acc;
}

}  // namespace vitocm
