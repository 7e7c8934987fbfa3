// Attention post-processing, thresholding and sliding-window stitching (HBM-bound byte/float
// work; warp-shuffle reductions, shared-memory histograms, no tensor cores):
//   head_mean_kernel        SSS/utils.py:232-233 + SSS/eval.py:142 / SSS/sw_processing.py:245,253-254
//   tile_threshold_kernel   SSS/eval.py:169-173 + SSS/utils.py:62-115 (per-image "ours"/otsu/heatmap masks)
//   extract_tiles_kernel    SSS/sw_processing.py:151-163 + ToTensor (:236-237)
//   stitch_gray_kernel      SSS/sw_processing.py:113-149 on the uint8 image crops (:225)
//   stitch_* kernels        SSS/sw_processing.py:255-259 (resize pair + concat_crops on the maps) and
//                           SSS/sw_processing.py:37-61 (global min-max, img*att, Otsu x2)
//   otsu_kernel             cv2.threshold(THRESH_OTSU) scan (OpenCV, restated in oracle/post_oracle.py)
#pragma once
#include "ptx.cuh"

namespace vitocm {

// order-preserving float <-> int map for atomicMin/atomicMax
__device__ __forceinline__ int f2ord(float f) {
  const int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float ord2f(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

// cv2.resize INTER_LINEAR source coordinate / weight for destination index d (scale = src/dst)
__device__ __forceinline__ void linear_coeff(int d, double scale, int src, int& s0, int& s1, float& f) {
  double fx = (d + 0.5) * scale - 0.5;
  int s = static_cast<int>(floor(fx));
  fx -= s;
  if (s < 0) { s = 0; fx = 0.0; }
  if (s >= src - 1) { s = src - 1; fx = 0.0; }
  s0 = s;
  s1 = min(s + 1, src - 1);
  f = static_cast<float>(fx);
}
// bilinear sample of a low-res map at full-res pixel (y, x): horizontal pass then vertical pass,
// fp32 with separate rounding of every product and sum (matches the numpy/cv2 oracle bit for bit)
__device__ __forceinline__ float bilinear_up(const float* __restrict__ lo, int lh, int lw, int y, int x, double scale) {
  int x0, x1, y0, y1;
  float fx, fy;
  linear_coeff(x, scale, lw, x0, x1, fx);
  linear_coeff(y, scale, lh, y0, y1, fy);
  const float a0 = __fsub_rn(1.0f, fx), b0 = __fsub_rn(1.0f, fy);
  const float r0 = __fadd_rn(__fmul_rn(lo[y0 * lw + x0], a0), __fmul_rn(lo[y0 * lw + x1], fx));
  const float r1 = __fadd_rn(__fmul_rn(lo[y1 * lw + x0], a0), __fmul_rn(lo[y1 * lw + x1], fx));
  return __fadd_rn(__fmul_rn(r0, b0), __fmul_rn(r1, fy));
}

// ---------------------------------------------------------------------------------------
// CLS rows [T][H][N] -> low-res map [T][n]: mean over heads of columns 1..N-1 (sequential fp32
// adds then a divide, as numpy reduces over a leading axis); mode 1 additionally applies the
// per-tile min-max * 255 of SSS/sw_processing.py:253-254.  One block per tile.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
head_mean_kernel(const float* __restrict__ rows, float* __restrict__ lowres, int heads, int N, int mode) {
  __shared__ float red_mn[8], red_mx[8];
  const int t = blockIdx.x, n = N - 1;
  const float* rt = rows + static_cast<long long>(t) * heads * N;
  float* lt = lowres + static_cast<long long>(t) * n;
  float mn = INFINITY, mx = -INFINITY;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float s = rt[1 + i];
    for (int h = 1; h < heads; ++h) s = __fadd_rn(s, rt[static_cast<long long>(h) * N + 1 + i]);
    s = __fdiv_rn(s, static_cast<float>(heads));
    lt[i] = s;
    mn = fminf(mn, s);
    mx = fmaxf(mx, s);
  }
  if (mode == 0) return;
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  mn = red_mn[0]; mx = red_mx[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) { mn = fminf(mn, red_mn[w]); mx = fmaxf(mx, red_mx[w]); }
  const float range = __fsub_rn(mx, mn);
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    lt[i] = __fmul_rn(__fdiv_rn(__fsub_rn(lt[i], mn), range), 255.0f);
}

// ---------------------------------------------------------------------------------------
// Cumulative-mass threshold of upstream DINO's visualize_attention.py, the semantics behind the reference's `--threshold`
// flag (help text at SSS/eval.py:33-34; the code itself is not under /root/reference: parity unpinned by the reference,
// oracle = oracle/post_oracle.py cummass_threshold).  Per (tile, head), over the n patch columns of the CLS row:
//     val, idx = sort(a) ascending;  val /= sum(val);  cum = cumsum(val);  keep = cum > 1 - th;  mask[idx] = keep
// i.e. the SMALLEST-attention patches holding 1 - th of the mass are dropped.  One block per (tile, head): bitonic sort of
// (value, index) pairs in shared memory (n padded to a power of two with +inf), row sum and inclusive scan by warp shuffles,
// scatter through the sorted indices; optionally the nearest x p upsampling (F.interpolate(mode="nearest")) as floats.
// ---------------------------------------------------------------------------------------
constexpr int CM_MAX = 4096;   // patches per tile (power of two bound): 224^2 / 8^2 = 784 -> 1024; 448^2 -> 3136 -> 4096
__global__ void __launch_bounds__(256)
cummass_kernel(const float* __restrict__ rows /*[T][H][N]*/, int heads, int N, int npow2, float keep_above /*fp32(1 - th)*/,
               uint8_t* __restrict__ mask /*[T][H][N-1]*/, float* __restrict__ up /*[T][H][lh*p][lw*p] or null*/, int lh, int lw, int p) {
  extern __shared__ float cm_smem[];           // val[npow2] | idx[npow2] (int) | warp partials[8]
  float* val = cm_smem;
  int* idx = reinterpret_cast<int*>(cm_smem + npow2);
  float* part = cm_smem + 2 * npow2;
  const int n = N - 1;
  const long long th_ = blockIdx.x;            // (tile, head) pair
  const float* a = rows + th_ * N + 1;         // skip the CLS column
  for (int i = threadIdx.x; i < npow2; i += blockDim.x) {
    val[i] = i < n ? a[i] : INFINITY;
    idx[i] = i;
  }
  __syncthreads();
  // bitonic sort ascending by (value, index)
  for (int k = 2; k <= npow2; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < npow2; i += blockDim.x) {
        const int l = i ^ j;
        if (l > i) {
          const bool up_dir = (i & k) == 0;
          const float vi = val[i], vl = val[l];
          const int ii = idx[i], il = idx[l];
          const bool gt = vi > vl || (vi == vl && ii > il);
          if (gt == up_dir) { val[i] = vl; val[l] = vi; idx[i] = il; idx[l] = ii; }
        }
      }
      __syncthreads();
    }
  }
  // total mass
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += val[i];
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  float total = 0.f;
  for (int w = 0; w < (blockDim.x >> 5); ++w) total += part[w];
  __syncthreads();
  // inclusive scan of val / total in sorted order: each thread owns a contiguous run of `per` elements
  const int per = (n + blockDim.x - 1) / blockDim.x;
  const int b0 = threadIdx.x * per, b1 = min(b0 + per, n);
  float run = 0.f;
  for (int i = b0; i < b1; ++i) run += __fdiv_rn(val[i], total);
  float incl = run;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 1; o < 32; o <<= 1) {
    const float t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) part[warp] = incl;
  __syncthreads();
  float base = incl - run;
  for (int w = 0; w < warp; ++w) base += part[w];
  uint8_t* m = mask + th_ * n;
  float c = base;
  for (int i = b0; i < b1; ++i) {
    c += __fdiv_rn(val[i], total);
    m[idx[i]] = c > keep_above ? 1 : 0;
  }
  if (up == nullptr) return;
  __syncthreads();                             // the mask row (global, written by this block) is read back below
  const int S = lw * p;
  float* u = up + th_ * static_cast<long long>(lh * p) * S;
  for (int i = threadIdx.x; i < lh * p * S; i += blockDim.x) {
    const int y = i / S, x = i - y * S;
    u[i] = static_cast<float>(m[(y / p) * lw + x / p]);
  }
}

// ---------------------------------------------------------------------------------------
// Otsu threshold from a 256-bin histogram (OpenCV's scan, fp64, first maximum wins).
// ---------------------------------------------------------------------------------------
__device__ inline int otsu_from_hist(const unsigned long long* hist) {
  double total = 0.0, wsum = 0.0;
  for (int i = 0; i < 256; ++i) { total += static_cast<double>(hist[i]); wsum += static_cast<double>(i) * static_cast<double>(hist[i]); }
  if (total <= 0.0) return 0;
  const double scale = 1.0 / total;
  const double mu = __dmul_rn(wsum, scale);
  double mu1 = 0.0, q1 = 0.0, max_sigma = 0.0;
  int max_val = 0;
  const double eps = 1.1920928955078125e-07;
  for (int i = 0; i < 256; ++i) {
    const double p_i = __dmul_rn(static_cast<double>(hist[i]), scale);
    mu1 = __dmul_rn(mu1, q1);
    q1 = __dadd_rn(q1, p_i);
    const double q2 = __dsub_rn(1.0, q1);
    if (fmin(q1, q2) < eps || fmax(q1, q2) > 1.0 - eps) continue;
    mu1 = __ddiv_rn(__dadd_rn(mu1, __dmul_rn(static_cast<double>(i), p_i)), q1);
    const double mu2 = __ddiv_rn(__dsub_rn(mu, __dmul_rn(q1, mu1)), q2);
    const double dm = __dsub_rn(mu1, mu2);
    const double sigma = __dmul_rn(__dmul_rn(__dmul_rn(q1, q2), dm), dm);
    if (sigma > max_sigma) { max_sigma = sigma; max_val = i; }
  }
  return max_val;
}

__global__ void otsu_kernel(const unsigned long long* __restrict__ hists, int nhist, int* __restrict__ thresholds) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nhist) thresholds[i] = otsu_from_hist(hists + static_cast<long long>(i) * 256);
}

// The same scan, one block of 256 threads per histogram (the mosaic path's three global histograms sit between two full-image
// passes: one thread walking 256 bins with two fp64 divisions each took 72 us).  Bit-identical to otsu_from_hist:
//   * total and the weighted sum add integers < 2^53: exact in any order -> tree reductions;
//   * p_i and i * p_i are independent per bin -> one thread each;
//   * the recurrence (mu1, q1) is OpenCV's and stays sequential in one thread, but carries ONE division per bin;
//   * mu2 / sigma of every bin in parallel, then "first bin with the greatest sigma > 0" as an (value, index) reduction.
__device__ __forceinline__ double otsu_block_sum(double v, double* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < 8; ++w) t += red[w];
  return t;
}
__global__ void __launch_bounds__(256) otsu_block_kernel(const unsigned long long* __restrict__ hists, int* __restrict__ thresholds) {
  __shared__ double p[256], ip[256], q1s[256], mu1s[256], red[8];
  __shared__ int valid[256];
  __shared__ double best_s[8];
  __shared__ int best_i[8];
  const int i = threadIdx.x;
  const double h = static_cast<double>(hists[static_cast<long long>(blockIdx.x) * 256 + i]);
  const double total = otsu_block_sum(h, red);
  const double wsum = otsu_block_sum(static_cast<double>(i) * h, red);
  if (total <= 0.0) {
    if (i == 0) thresholds[blockIdx.x] = 0;
    return;
  }
  const double scale = 1.0 / total;
  const double mu = __dmul_rn(wsum, scale);
  const double p_i = __dmul_rn(h, scale);
  p[i] = p_i;
  ip[i] = __dmul_rn(static_cast<double>(i), p_i);
  __syncthreads();
  if (i == 0) {
    const double eps = 1.1920928955078125e-07;
    double mu1 = 0.0, q1 = 0.0;
    for (int k = 0; k < 256; ++k) {
      mu1 = __dmul_rn(mu1, q1);
      q1 = __dadd_rn(q1, p[k]);
      const double q2 = __dsub_rn(1.0, q1);
      if (fmin(q1, q2) < eps || fmax(q1, q2) > 1.0 - eps) { valid[k] = 0; continue; }
      mu1 = __ddiv_rn(__dadd_rn(mu1, ip[k]), q1);
      q1s[k] = q1;
      mu1s[k] = mu1;
      valid[k] = 1;
    }
  }
  __syncthreads();
  double sigma = -1.0;
  if (valid[i]) {
    const double q1 = q1s[i], mu1 = mu1s[i];
    const double q2 = __dsub_rn(1.0, q1);
    const double mu2 = __ddiv_rn(__dsub_rn(mu, __dmul_rn(q1, mu1)), q2);
    const double dm = __dsub_rn(mu1, mu2);
    sigma = __dmul_rn(__dmul_rn(__dmul_rn(q1, q2), dm), dm);
    if (!(sigma > 0.0)) sigma = -1.0;   // the scan only accepts sigma > max_sigma >= 0 (NaN never wins)
  }
  int idx = i;
  for (int o = 16; o > 0; o >>= 1) {
    const double s2 = __shfl_xor_sync(0xffffffffu, sigma, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, idx, o);
    if (s2 > sigma || (s2 == sigma && i2 < idx)) { sigma = s2; idx = i2; }
  }
  if ((i & 31) == 0) { best_s[i >> 5] = sigma; best_i[i >> 5] = idx; }
  __syncthreads();
  if (i == 0) {
    for (int w = 1; w < 8; ++w)
      if (best_s[w] > sigma || (best_s[w] == sigma && best_i[w] < idx)) { sigma = best_s[w]; idx = best_i[w]; }
    thresholds[blockIdx.x] = sigma > 0.0 ? idx : 0;
  }
}

// ---------------------------------------------------------------------------------------
// Per-image threshold (eval / PGT flavour).  One block per tile, three passes over the tile:
//   1. att = bilinear_up(lowres) ; block min / max
//   2. att_u8 = trunc((att-min)/(max-min)*255) ; result = trunc((img/2)*0.6 + (att_u8/2)*0.4) (fp64)
//      -> three 256-bin histograms (result, img, att_u8) in shared memory -> Otsu x3
//   3. masks th / th2 / th3
// img = PIL "L" of ToPILImage(x): floor(x*255) per channel, then (19595 R + 38470 G + 7471 B + 32768) >> 16.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int gray_u8_from_x(const float* __restrict__ xt, int C, long long plane, long long off) {
  const int r = static_cast<int>(xt[off] * 255.0f);
  if (C < 3) return r;
  const int g = static_cast<int>(xt[plane + off] * 255.0f);
  const int b = static_cast<int>(xt[2 * plane + off] * 255.0f);
  return (19595 * r + 38470 * g + 7471 * b + 0x8000) >> 16;
}

__global__ void __launch_bounds__(512)
tile_threshold_kernel(const float* __restrict__ lowres /*[T][lh][lw]*/, const float* __restrict__ x /*[T][C][S][S]*/,
                      int C, int S, int lh, int lw, uint8_t* __restrict__ masks /*[T][3][S][S]*/,
                      int* __restrict__ thresholds /*[T][3]*/, float* __restrict__ att_out /*[T][S][S] or null*/,
                      const float* __restrict__ att_in /*[T][S][S] or null: use instead of upsampling lowres*/,
                      const uint8_t* __restrict__ img_in /*[T][S][S] or null: use instead of deriving from x*/,
                      uint8_t* __restrict__ aux /*[T][2][S][S] or null: the blended image `result` and att_u8 (the images utils.threshold saves)*/) {
  __shared__ float red_mn[16], red_mx[16];
  __shared__ unsigned int hist[3][256];
  __shared__ unsigned long long hist64[256];
  __shared__ int thr[3];
  const int t = blockIdx.x;
  const float* lo = lowres + static_cast<long long>(t) * lh * lw;
  const long long plane = static_cast<long long>(S) * S;
  const float* xt = x + static_cast<long long>(t) * C * plane;
  const float* ain = att_in != nullptr ? att_in + static_cast<long long>(t) * plane : nullptr;
  const uint8_t* iin = img_in != nullptr ? img_in + static_cast<long long>(t) * plane : nullptr;
  const double scale = static_cast<double>(lw) / static_cast<double>(S);
  const int npx = S * S;
  float mn = INFINITY, mx = -INFINITY;
  for (int i = threadIdx.x; i < npx; i += blockDim.x) {
    const float a = ain != nullptr ? ain[i] : bilinear_up(lo, lh, lw, i / S, i % S, scale);
    if (att_out != nullptr) att_out[static_cast<long long>(t) * plane + i] = a;
    mn = fminf(mn, a);
    mx = fmaxf(mx, a);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; }
  for (int i = threadIdx.x; i < 3 * 256; i += blockDim.x) (&hist[0][0])[i] = 0u;
  __syncthreads();
  mn = red_mn[0]; mx = red_mx[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) { mn = fminf(mn, red_mn[w]); mx = fmaxf(mx, red_mx[w]); }
  const bool flat = (mx == mn);  // min_max_normalize returns its input when the map is flat
  const float range = __fsub_rn(mx, mn);
  auto classify = [&](int i, int& img, int& att_u8, int& res) {
    const float a = ain != nullptr ? ain[i] : bilinear_up(lo, lh, lw, i / S, i % S, scale);
    const float an = flat ? a : __fdiv_rn(__fsub_rn(a, mn), range);
    att_u8 = static_cast<int>(static_cast<uint8_t>(static_cast<int>(__fmul_rn(an, 255.0f))));
    img = iin != nullptr ? static_cast<int>(iin[i]) : gray_u8_from_x(xt, C, plane, i);
    const double r = __dadd_rn(__dmul_rn(static_cast<double>(img) / 2.0, 1.0 - 0.4), __dmul_rn(static_cast<double>(att_u8) / 2.0, 0.4));
    res = static_cast<int>(r);
  };
  for (int i = threadIdx.x; i < npx; i += blockDim.x) {
    int img, au, res;
    classify(i, img, au, res);
    atomicAdd(&hist[0][res], 1u);
    atomicAdd(&hist[1][img], 1u);
    atomicAdd(&hist[2][au], 1u);
  }
  __syncthreads();
  for (int k = 0; k < 3; ++k) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist64[i] = hist[k][i];
    __syncthreads();
    if (threadIdx.x == 0) {
      thr[k] = otsu_from_hist(hist64);
      thresholds[t * 3 + k] = thr[k];
    }
    __syncthreads();
  }
  uint8_t* m0 = masks + static_cast<long long>(t) * 3 * plane;
  for (int i = threadIdx.x; i < npx; i += blockDim.x) {
    int img, au, res;
    classify(i, img, au, res);
    m0[i] = res > thr[0] ? 255 : 0;
    m0[plane + i] = img > thr[1] ? 255 : 0;
    m0[2 * plane + i] = au > thr[2] ? 255 : 0;
    if (aux != nullptr) {
      aux[static_cast<long long>(t) * 2 * plane + i] = static_cast<uint8_t>(res);
      aux[static_cast<long long>(t) * 2 * plane + plane + i] = static_cast<uint8_t>(au);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Ragged forms for images of different sizes packed back to back (vitocm_forward_cls_attn_varlen's layout), one block per image:
//   head_mean_var_kernel       head_mean_kernel with image t's rows [H][N_t] at heads (patch_off[t] + t) and its map at patch_off[t]
//   tile_threshold_var_kernel  tile_threshold_kernel (without att_in / img_in / aux) for a square image of side S_t = geo[t].x
//                              and map side geo[t].y, map at geo[t].z, pixels at geo[t].w (x: C x, masks: 3 x)
// The per-image arithmetic is the uniform kernels' own.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
head_mean_var_kernel(const float* __restrict__ rows, float* __restrict__ lowres, int heads, const int* __restrict__ patch_off, int mode) {
  __shared__ float red_mn[8], red_mx[8];
  const int t = blockIdx.x, p0 = patch_off[t], n = patch_off[t + 1] - p0, N = n + 1;
  const float* rt = rows + static_cast<long long>(p0 + t) * heads;
  float* lt = lowres + p0;
  float mn = INFINITY, mx = -INFINITY;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float s = rt[1 + i];
    for (int h = 1; h < heads; ++h) s = __fadd_rn(s, rt[static_cast<long long>(h) * N + 1 + i]);
    s = __fdiv_rn(s, static_cast<float>(heads));
    lt[i] = s;
    mn = fminf(mn, s);
    mx = fmaxf(mx, s);
  }
  if (mode == 0) return;
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  mn = red_mn[0]; mx = red_mx[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) { mn = fminf(mn, red_mn[w]); mx = fmaxf(mx, red_mx[w]); }
  const float range = __fsub_rn(mx, mn);
  for (int i = threadIdx.x; i < n; i += blockDim.x)
    lt[i] = __fmul_rn(__fdiv_rn(__fsub_rn(lt[i], mn), range), 255.0f);
}

__global__ void __launch_bounds__(512)
tile_threshold_var_kernel(const float* __restrict__ lowres, const float* __restrict__ x, int C, const int4* __restrict__ geo,
                          uint8_t* __restrict__ masks, int* __restrict__ thresholds, float* __restrict__ att_out) {
  __shared__ float red_mn[16], red_mx[16];
  __shared__ unsigned int hist[3][256];
  __shared__ unsigned long long hist64[256];
  __shared__ int thr[3];
  const int t = blockIdx.x;
  const int4 g = geo[t];
  const int S = g.x, lh = g.y, lw = g.y;
  const float* lo = lowres + g.z;
  const long long plane = static_cast<long long>(S) * S;
  const float* xt = x + static_cast<long long>(g.w) * C;
  const double scale = static_cast<double>(lw) / static_cast<double>(S);
  const int npx = S * S;
  float mn = INFINITY, mx = -INFINITY;
  for (int i = threadIdx.x; i < npx; i += blockDim.x) {
    const float a = bilinear_up(lo, lh, lw, i / S, i % S, scale);
    if (att_out != nullptr) att_out[g.w + i] = a;
    mn = fminf(mn, a);
    mx = fmaxf(mx, a);
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; }
  for (int i = threadIdx.x; i < 3 * 256; i += blockDim.x) (&hist[0][0])[i] = 0u;
  __syncthreads();
  mn = red_mn[0]; mx = red_mx[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) { mn = fminf(mn, red_mn[w]); mx = fmaxf(mx, red_mx[w]); }
  const bool flat = (mx == mn);
  const float range = __fsub_rn(mx, mn);
  auto classify = [&](int i, int& img, int& att_u8, int& res) {
    const float a = bilinear_up(lo, lh, lw, i / S, i % S, scale);
    const float an = flat ? a : __fdiv_rn(__fsub_rn(a, mn), range);
    att_u8 = static_cast<int>(static_cast<uint8_t>(static_cast<int>(__fmul_rn(an, 255.0f))));
    img = gray_u8_from_x(xt, C, plane, i);
    const double r = __dadd_rn(__dmul_rn(static_cast<double>(img) / 2.0, 1.0 - 0.4), __dmul_rn(static_cast<double>(att_u8) / 2.0, 0.4));
    res = static_cast<int>(r);
  };
  for (int i = threadIdx.x; i < npx; i += blockDim.x) {
    int img, au, res;
    classify(i, img, au, res);
    atomicAdd(&hist[0][res], 1u);
    atomicAdd(&hist[1][img], 1u);
    atomicAdd(&hist[2][au], 1u);
  }
  __syncthreads();
  for (int k = 0; k < 3; ++k) {
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist64[i] = hist[k][i];
    __syncthreads();
    if (threadIdx.x == 0) {
      thr[k] = otsu_from_hist(hist64);
      thresholds[t * 3 + k] = thr[k];
    }
    __syncthreads();
  }
  uint8_t* m0 = masks + static_cast<long long>(g.w) * 3;
  for (int i = threadIdx.x; i < npx; i += blockDim.x) {
    int img, au, res;
    classify(i, img, au, res);
    m0[i] = res > thr[0] ? 255 : 0;
    m0[plane + i] = img > thr[1] ? 255 : 0;
    m0[2 * plane + i] = au > thr[2] ? 255 : 0;
  }
}

// ---------------------------------------------------------------------------------------
// Sliding-window geometry shared by the mosaic kernels.  ny x nx tiles of size W at stride S
// (origins range(0, size - 2S, S) over the height and over the width), row-major: tile t = i * nx + j has origin (i S, j S);
// stitched extent Ey x Ex = ((ny-1) S + W) x ((nx-1) S + W); step = W - S.  A square mosaic is ny = nx = n.
// wtab[k] = numpy.linspace(1, 0, step)[k] (computed on the host so it is bit-identical).
// ---------------------------------------------------------------------------------------
struct StitchGeom {
  int ny, nx, W, S, step, Ey, Ex;
  int lh, lw;        // low-res map size (W / patch)
  double scale;      // lw / W
};

// sliding_window + ToTensor: mosaic u8 gray [mos_h][pitch] -> x [T][C][W][W] fp32 = v / 255 (zero padded
// outside the mosaic like PIL's crop); tiles t0 .. t0+T-1 in row-major order of a grid nx windows wide.
__global__ void extract_tiles_kernel(const uint8_t* __restrict__ mosaic, int mos_h, int mos_w, long long pitch, int nx,
                                     int W, int S, int t0, int T, int C, float* __restrict__ x) {
  const long long per_tile = static_cast<long long>(W) * W;
  const long long total = per_tile * T;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int tl = static_cast<int>(i / per_tile);
    const int r = static_cast<int>(i - tl * per_tile);
    const int y = r / W, xx = r - y * W;
    const int t = t0 + tl;
    const int gy = (t / nx) * S + y, gx = (t % nx) * S + xx;
    const float v = (gy < mos_h && gx < mos_w) ? __fdiv_rn(static_cast<float>(mosaic[gy * pitch + gx]), 255.0f) : 0.f;
    float* xt = x + static_cast<long long>(tl) * C * per_tile + r;
    for (int c = 0; c < C; ++c) xt[c * per_tile] = v;
  }
}

// uint8 blend of the image crops: sequential pairwise blend with truncation, first along x inside
// each strip, then along y across strips -- what concat_crops does to the uint8 crops at :225.
__device__ __forceinline__ uint8_t blend_u8(uint8_t a, uint8_t b, double w) {
  return static_cast<uint8_t>(static_cast<int>(__dadd_rn(__dmul_rn(static_cast<double>(a), w), __dmul_rn(static_cast<double>(b), __dsub_rn(1.0, w)))));
}
// Row-organised: a thread owns V consecutive pixels of a row; the covering-tile ranges come from one division per thread,
// the vertical blend sequence (same for the whole row) from the row index.
template <int V>
__global__ void __launch_bounds__(256)
stitch_gray_kernel(const uint8_t* __restrict__ mosaic, int mos_h, int mos_w, long long pitch, StitchGeom g,
                   const double* __restrict__ wtab, int y_begin, int y_end, uint8_t* __restrict__ out /*[Ey][Ex]*/) {
  const int X0 = (blockIdx.x * 256 + threadIdx.x) * V;
  if (X0 >= g.Ex) return;
  const int dW = g.W / g.S, eW = g.W % g.S;
  const int q0 = X0 / g.S, r0 = X0 - q0 * g.S;
  for (int Y = y_begin + blockIdx.y; Y < y_end; Y += gridDim.y) {
    const int qy = Y / g.S, ry = Y - qy * g.S;
    int i1 = min(qy, g.ny - 1);
    int i0 = qy + 1 - dW - (ry < eW ? 1 : 0);
    if (i0 < 0) i0 = 0;
    uint8_t res[V];
    int q = q0, r = r0;
#pragma unroll
    for (int u = 0; u < V; ++u) {
      const int X = X0 + u;
      // every crop holds the same source pixel (zero beyond the mosaic)
      const uint8_t src = (Y < mos_h && X < mos_w) ? __ldg(mosaic + Y * pitch + X) : 0;
      int j1 = min(q, g.nx - 1);
      int j0 = q + 1 - dW - (r < eW ? 1 : 0);
      if (j0 < 0) j0 = 0;
      // horizontal sequence is identical for every strip (same source value)
      uint8_t hv = src;
      for (int j = j0 + 1; j <= j1; ++j) {
        const int kx = (q - j) * g.S + r;
        hv = (kx < g.step) ? blend_u8(hv, src, __ldg(wtab + kx)) : src;
      }
      uint8_t v = hv;
      for (int i = i0 + 1; i <= i1; ++i) {
        const int ky = Y - i * g.S;
        v = (ky < g.step) ? blend_u8(v, hv, __ldg(wtab + ky)) : hv;
      }
      res[u] = v;
      if (++r == g.S) { r = 0; ++q; }
    }
    const long long o = static_cast<long long>(Y) * g.Ex + X0;
    if (V == 4) *reinterpret_cast<uchar4*>(out + o) = make_uchar4(res[0], res[1 % V], res[2 % V], res[3 % V]);
    else out[o] = res[0];
  }
}

// tiles covering coordinate P = q * S + r (q = P / S) along an axis of `cnt` tiles: [c0, c1]
__device__ __forceinline__ void cover_range(int cnt, int q, int r, int dW, int eW, int& c0, int& c1) {
  c1 = min(q, cnt - 1);
  c0 = q + 1 - dW - (r < eW ? 1 : 0);      // = (P - W + S) / S for P >= W - S ... clamped below
  if (c0 < 0) c0 = 0;
}

// Column-strip form of stitch_gray_kernel (same structure as stitch_strip_kernel below): a thread owns V adjacent columns over a
// band of SC_ROWS consecutive rows; its horizontal blend weights are computed once, the vertical ones once per row by one thread.
// Same blend sequence per pixel (bit-identical); the row-organised kernel re-derived both per pixel (~100 instructions).
constexpr int SG_THREADS = 256;
constexpr int SG_ROWS = 32;
__device__ __forceinline__ uint8_t blend_u8_pre(uint8_t a, uint8_t b, double w, double omw) {   // blend_u8 with 1 - w precomputed
  return static_cast<uint8_t>(static_cast<int>(__dadd_rn(__dmul_rn(static_cast<double>(a), w), __dmul_rn(static_cast<double>(b), omw))));
}
template <int V, int MC>
__global__ void __launch_bounds__(SG_THREADS)
stitch_gray_strip_kernel(const uint8_t* __restrict__ mosaic, int mos_h, int mos_w, long long pitch, StitchGeom g,
                         const double* __restrict__ wtab, int y_begin, int y_end, uint8_t* __restrict__ out /*[Ey][Ex]*/) {
  constexpr int NS = MC - 1;   // blend steps per direction
  __shared__ int s_n[SG_ROWS];
  __shared__ int s_bl[SG_ROWS][NS];
  __shared__ double s_w[SG_ROWS][NS], s_omw[SG_ROWS][NS];
  const int yb = y_begin + blockIdx.y * SG_ROWS;
  const int nrows = min(SG_ROWS, y_end - yb);
  const int dW = g.W / g.S, eW = g.W % g.S;
  if (static_cast<int>(threadIdx.x) < nrows) {
    const int Y = yb + threadIdx.x;
    const int qy = Y / g.S, ry = Y - qy * g.S;
    int i0, i1;
    cover_range(g.ny, qy, ry, dW, eW, i0, i1);
    int nb = i1 - i0;
    if (nb > NS) nb = NS;
    s_n[threadIdx.x] = nb;
#pragma unroll
    for (int s2 = 0; s2 < NS; ++s2) {
      if (s2 < nb) {
        const int ky = Y - (i0 + 1 + s2) * g.S;
        const int bl = ky < g.step ? 1 : 0;
        const double w = bl ? wtab[ky] : 0.0;
        s_bl[threadIdx.x][s2] = bl;
        s_w[threadIdx.x][s2] = w;
        s_omw[threadIdx.x][s2] = __dsub_rn(1.0, w);
      }
    }
  }
  __syncthreads();
  const int X0 = (blockIdx.x * SG_THREADS + threadIdx.x) * V;
  if (X0 >= g.Ex) return;
  int nbx[V], blx[V][NS];
  double wx[V][NS], omwx[V][NS];
  {
    int q = X0 / g.S, r = X0 - q * g.S;
#pragma unroll
    for (int u = 0; u < V; ++u) {
      int j0, j1;
      cover_range(g.nx, q, r, dW, eW, j0, j1);
      nbx[u] = min(j1 - j0, NS);
#pragma unroll
      for (int s2 = 0; s2 < NS; ++s2) {
        blx[u][s2] = 0; wx[u][s2] = 0.0; omwx[u][s2] = 1.0;
        if (s2 < nbx[u]) {
          const int kx = (q - (j0 + 1 + s2)) * g.S + r;
          blx[u][s2] = kx < g.step ? 1 : 0;
          wx[u][s2] = blx[u][s2] ? wtab[kx] : 0.0;
          omwx[u][s2] = __dsub_rn(1.0, wx[u][s2]);
        }
      }
      if (++r == g.S) { r = 0; ++q; }
    }
  }
  const bool vec_in = V == 4 && X0 + 4 <= mos_w && ((reinterpret_cast<uintptr_t>(mosaic) | static_cast<uintptr_t>(pitch)) & 3) == 0;
  for (int t = 0; t < nrows; ++t) {
    const int Y = yb + t;
    uint8_t src[V];
    if (Y < mos_h && vec_in) {
      const uchar4 b = *reinterpret_cast<const uchar4*>(mosaic + Y * pitch + X0);
      src[0] = b.x; src[1 % V] = b.y; src[2 % V] = b.z; src[3 % V] = b.w;
    } else {
#pragma unroll
      for (int u = 0; u < V; ++u) src[u] = (Y < mos_h && X0 + u < mos_w) ? __ldg(mosaic + Y * pitch + X0 + u) : 0;   // zero beyond the mosaic
    }
    const int nb = s_n[t];
    uint8_t res[V];
#pragma unroll
    for (int u = 0; u < V; ++u) {
      uint8_t hv = src[u];   // every crop holds the same source pixel: the horizontal sequence is identical for every strip
#pragma unroll
      for (int s2 = 0; s2 < NS; ++s2)
        if (s2 < nbx[u]) hv = blx[u][s2] ? blend_u8_pre(hv, src[u], wx[u][s2], omwx[u][s2]) : src[u];
      uint8_t v = hv;
#pragma unroll
      for (int s2 = 0; s2 < NS; ++s2)
        if (s2 < nb) v = s_bl[t][s2] ? blend_u8_pre(v, hv, s_w[t][s2], s_omw[t][s2]) : hv;
      res[u] = v;
    }
    const long long o = static_cast<long long>(Y) * g.Ex + X0;
    if (V == 4) *reinterpret_cast<uchar4*>(out + o) = make_uchar4(res[0], res[1 % V], res[2 % V], res[3 % V]);
    else out[o] = res[0];
  }
}

// value of the stitched attention map at (Y, X): sequential blends of the bilinearly upsampled
// per-tile maps, fp64 products/sum rounded to fp32 at every seam (the crops are float32 arrays).
__device__ __forceinline__ float blend_f32(float a, float b, double w) {
  return static_cast<float>(__dadd_rn(__dmul_rn(static_cast<double>(a), w), __dmul_rn(static_cast<double>(b), __dsub_rn(1.0, w))));
}
__device__ __forceinline__ float stitched_value(const float* __restrict__ lowres, const StitchGeom& g,
                                                const double* __restrict__ wtab, int Y, int X) {
  int j0 = (X - g.W + g.S) / g.S; if (X - g.W + 1 <= 0) j0 = 0; if (j0 < 0) j0 = 0;
  const int j1 = min(X / g.S, g.nx - 1);
  int i0 = (Y - g.W + g.S) / g.S; if (Y - g.W + 1 <= 0) i0 = 0; if (i0 < 0) i0 = 0;
  const int i1 = min(Y / g.S, g.ny - 1);
  const int lsz = g.lh * g.lw;
  float v = 0.f;
  for (int i = i0; i <= i1; ++i) {
    const int ky = Y - i * g.S;
    float hv = 0.f;
    for (int j = j0; j <= j1; ++j) {
      const int kx = X - j * g.S;
      const float tv = bilinear_up(lowres + static_cast<long long>(i * g.nx + j) * lsz, g.lh, g.lw, ky, kx, g.scale);
      hv = (j > j0 && kx < g.step) ? blend_f32(hv, tv, wtab[kx]) : tv;
    }
    v = (i > i0 && ky < g.step) ? blend_f32(v, hv, wtab[ky]) : hv;
  }
  return v;
}

// concat_crops (SSS/sw_processing.py:113-134) on full-resolution float32 crops [ny*nx][W][W] -> out [Ey][Ex]
__global__ void concat_crops_f32_kernel(const float* __restrict__ crops, StitchGeom g, const double* __restrict__ wtab,
                                        float* __restrict__ out) {
  const long long total = static_cast<long long>(g.Ey) * g.Ex;
  const long long tsz = static_cast<long long>(g.W) * g.W;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int Y = static_cast<int>(idx / g.Ex), X = static_cast<int>(idx % g.Ex);
    int j0 = (X - g.W + g.S) / g.S; if (X - g.W + 1 <= 0) j0 = 0;
    const int j1 = min(X / g.S, g.nx - 1);
    int i0 = (Y - g.W + g.S) / g.S; if (Y - g.W + 1 <= 0) i0 = 0;
    const int i1 = min(Y / g.S, g.ny - 1);
    float v = 0.f;
    for (int i = i0; i <= i1; ++i) {
      const int ky = Y - i * g.S;
      float hv = 0.f;
      for (int j = j0; j <= j1; ++j) {
        const int kx = X - j * g.S;
        const float tv = crops[(i * g.nx + j) * tsz + static_cast<long long>(ky) * g.W + kx];
        hv = (j > j0 && kx < g.step) ? blend_f32(hv, tv, wtab[kx]) : tv;
      }
      v = (i > i0 && ky < g.step) ? blend_f32(v, hv, wtab[ky]) : hv;
    }
    out[idx] = v;
  }
}
// same on uint8 crops [ny*nx][W][W][C] (HWC, as PIL / numpy image crops) -> out [Ey][Ex][C]
__global__ void concat_crops_u8_kernel(const uint8_t* __restrict__ crops, StitchGeom g, int C, const double* __restrict__ wtab,
                                       uint8_t* __restrict__ out) {
  const long long total = static_cast<long long>(g.Ey) * g.Ex * C;
  const long long tsz = static_cast<long long>(g.W) * g.W * C;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const long long px = idx / C;
    const int Y = static_cast<int>(px / g.Ex), X = static_cast<int>(px % g.Ex);
    int j0 = (X - g.W + g.S) / g.S; if (X - g.W + 1 <= 0) j0 = 0;
    const int j1 = min(X / g.S, g.nx - 1);
    int i0 = (Y - g.W + g.S) / g.S; if (Y - g.W + 1 <= 0) i0 = 0;
    const int i1 = min(Y / g.S, g.ny - 1);
    uint8_t v = 0;
    for (int i = i0; i <= i1; ++i) {
      const int ky = Y - i * g.S;
      uint8_t hv = 0;
      for (int j = j0; j <= j1; ++j) {
        const int kx = X - j * g.S;
        const uint8_t tv = crops[(i * g.nx + j) * tsz + (static_cast<long long>(ky) * g.W + kx) * C + c];
        hv = (j > j0 && kx < g.step) ? blend_u8(hv, tv, wtab[kx]) : tv;
      }
      v = (i > i0 && ky < g.step) ? blend_u8(v, hv, wtab[ky]) : hv;
    }
    out[idx] = v;
  }
}
// sliding_window on a uint8 HWC image -> crops [ny*nx][W][W][C], zero padded outside the image.
// Window (iy, ix) starts at (oy[iy], ox[ix]) = (iy*S, ix*S).
__global__ void crop_u8_kernel(const uint8_t* __restrict__ img, int img_h, int img_w, int C, int ny, int nx, int W, int S,
                               uint8_t* __restrict__ crops) {
  const long long tsz = static_cast<long long>(W) * W * C;
  const long long total = tsz * ny * nx;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int t = static_cast<int>(idx / tsz);
    const long long r = idx - t * tsz;
    const int c = static_cast<int>(r % C);
    const int xx = static_cast<int>((r / C) % W), yy = static_cast<int>(r / (static_cast<long long>(C) * W));
    const int gy = (t / nx) * S + yy, gx = (t % nx) * S + xx;
    crops[idx] = (gy < img_h && gx < img_w) ? img[(static_cast<long long>(gy) * img_w + gx) * C + c] : 0;
  }
}

// ---------------------------------------------------------------------------------------
// Crop variants of the eval / analyse scripts (SURVEY.md 8f rank 3).
// ---------------------------------------------------------------------------------------
// concat_crops_overlap(crops, stride) (SSS/utils.py:319-347): n x n crops of size W overlapping by
// V = 2 * stride; inside an overlap the running image and the next crop are each floor-halved and added
// (`a // 2 + b // 2`), first along x inside a strip, then along y across strips -- except that the LAST
// strip is appended without blending: its overlap rows keep the running image (:337-339).
// Gather form: the value of an output pixel is the fold, in crop order, over the crops that cover it.
struct OverlapGeom {
  int n, W, V, step, E;   // step = W - V, E = W + (n-1) * step
};
__device__ __forceinline__ float half_floor(float a) { return floorf(__fmul_rn(a, 0.5f)); }
__device__ __forceinline__ float avg_halves(float a, float b) { return __fadd_rn(half_floor(a), half_floor(b)); }
__device__ __forceinline__ uint8_t avg_halves(uint8_t a, uint8_t b) { return static_cast<uint8_t>((a >> 1) + (b >> 1)); }

template <typename T>
__global__ void concat_crops_overlap_kernel(const T* __restrict__ crops /*[n*n][W][W][C]*/, OverlapGeom g, int C,
                                            T* __restrict__ out /*[E][E][C]*/) {
  const long long total = static_cast<long long>(g.E) * g.E * C;
  const long long tsz = static_cast<long long>(g.W) * g.W * C;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(idx % C);
    const long long px = idx / C;
    const int Y = static_cast<int>(px / g.E), X = static_cast<int>(px % g.E);
    // crops covering X: j*step <= X < j*step + W
    int j0 = X < g.W ? 0 : (X - g.W) / g.step + 1;
    const int j1 = min(X / g.step, g.n - 1);
    int i0 = Y < g.W ? 0 : (Y - g.W) / g.step + 1;
    const int i1 = min(Y / g.step, g.n - 1);
    T v = T(0);
    for (int i = i0; i <= i1; ++i) {
      const int ky = Y - i * g.step;
      T hv = T(0);
      for (int j = j0; j <= j1; ++j) {
        const int kx = X - j * g.step;
        const T tv = crops[(i * g.n + j) * tsz + (static_cast<long long>(ky) * g.W + kx) * C + c];
        hv = (j > j0 && kx < g.V) ? avg_halves(hv, tv) : tv;
      }
      if (i > i0 && ky < g.V) {
        if (i != g.n - 1) v = avg_halves(v, hv);   // last strip: the running image is kept as it is
      } else {
        v = hv;
      }
    }
    out[idx] = v;
  }
}

// plain n x n tiling (SSS/utils.py:304-317 `concat_crops`; SSS/eval.py:160-161) of one channel of batched crops:
// src [B][cr*cr][C][h][w] fp32 -> dst [B][cr*h][cr*w], channel c0.  Pure data movement.
__global__ void concat_grid_f32_kernel(const float* __restrict__ src, int B, int cr, int C, int c0, int h, int w,
                                       float* __restrict__ dst) {
  const int EH = cr * h, EW = cr * w;
  const long long total = static_cast<long long>(B) * EH * EW;
  for (long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int X = static_cast<int>(idx % EW);
    const int Y = static_cast<int>((idx / EW) % EH);
    const int b = static_cast<int>(idx / (static_cast<long long>(EW) * EH));
    const int ci = Y / h, cj = X / w;
    dst[idx] = src[(((static_cast<long long>(b) * cr * cr + ci * cr + cj) * C + c0) * h + (Y - ci * h)) * w + (X - cj * w)];
  }
}

// ---------------------------------------------------------------------------------------
// Row-organised mosaic passes (round 2).  The first versions of these kernels walked a flat pixel index (two 64-bit divisions
// per pixel), moved one byte per thread and re-evaluated the stitched map -- <= 4 bilinear samples and 3 fp64 blends per pixel --
// in all three passes: 1.4 ms per 4032^2 mosaic, ~0.6 % of the HBM roofline.  Now a block owns 256*V consecutive pixels of a
// row (V = 4 when rows are 16-byte aligned), everything that depends on the row only (covering tile rows, vertical bilinear
// coefficients, vertical blend weights) is computed once per row, the horizontal coefficients come from a per-block table,
// accesses are float4 / uchar4, and the stitched map is evaluated ONCE (pass 1 stores it as fp32, passes 2 and 3 stream it
// back, mostly out of the 126 MB L2).  The arithmetic per value is unchanged (bilinear_tab == bilinear_up, blend_f32,
// sw_classify), so the outputs stay bit-identical to the reference's sequential loops.
// ---------------------------------------------------------------------------------------
constexpr int ST_THREADS = 256;
constexpr int ST_MAX_W = 1024;          // per-block coefficient table: W entries

struct LinTab { int s0, s1; float f; };

__device__ __forceinline__ float bilinear_tab(const float* __restrict__ lo, int lw, int y0, int y1, float fy, int x0, int x1, float fx) {
  const float a0 = __fsub_rn(1.0f, fx), b0 = __fsub_rn(1.0f, fy);
  const float r0 = __fadd_rn(__fmul_rn(__ldg(lo + y0 * lw + x0), a0), __fmul_rn(__ldg(lo + y0 * lw + x1), fx));
  const float r1 = __fadd_rn(__fmul_rn(__ldg(lo + y1 * lw + x0), a0), __fmul_rn(__ldg(lo + y1 * lw + x1), fx));
  return __fadd_rn(__fmul_rn(r0, b0), __fmul_rn(r1, fy));
}

// stitched value at (row context, X): same evaluation order as stitched_value()
struct RowCtx {
  int i0, i1;
  int ky[4], y0[4], y1[4];
  float fy[4];
};
__device__ __forceinline__ void make_row_ctx(const StitchGeom& g, int Y, RowCtx& rc) {
  const int q = Y / g.S, r = Y - q * g.S;
  cover_range(g.ny, q, r, g.W / g.S, g.W % g.S, rc.i0, rc.i1);
  if (rc.i1 - rc.i0 > 3) rc.i1 = rc.i0 + 3;   // (host guarantees W <= 4 S)
  for (int k = 0; k <= rc.i1 - rc.i0; ++k) {
    rc.ky[k] = Y - (rc.i0 + k) * g.S;
    linear_coeff(rc.ky[k], g.scale, g.lh, rc.y0[k], rc.y1[k], rc.fy[k]);
  }
}
__device__ __forceinline__ float stitched_value_row(const float* __restrict__ lowres, const StitchGeom& g, const double* __restrict__ wtab,
                                                    const LinTab* __restrict__ tab, const RowCtx& rc, int q, int r, int dW, int eW) {
  int j0, j1;
  cover_range(g.nx, q, r, dW, eW, j0, j1);
  const int lsz = g.lh * g.lw;
  float v = 0.f;
  for (int k = 0; k <= rc.i1 - rc.i0; ++k) {
    const int i = rc.i0 + k;
    float hv = 0.f;
    for (int j = j0; j <= j1; ++j) {
      const int kx = (q - j) * g.S + r;
      const LinTab t = tab[kx];
      const float tv = bilinear_tab(lowres + static_cast<long long>(i * g.nx + j) * lsz, g.lw, rc.y0[k], rc.y1[k], rc.fy[k], t.s0, t.s1, t.f);
      hv = (j > j0 && kx < g.step) ? blend_f32(hv, tv, __ldg(wtab + kx)) : tv;
    }
    v = (k > 0 && rc.ky[k] < g.step) ? blend_f32(v, hv, __ldg(wtab + rc.ky[k])) : hv;
  }
  return v;
}

// launch geometry: grid.x covers a row in groups of 256 * V pixels, grid.y strides over the rows of the band
template <int V>
__device__ __forceinline__ int st_x0() { return (blockIdx.x * ST_THREADS + threadIdx.x) * V; }

// pass 1: stitched map of rows [y_begin, y_end) -> map_out (fp32, absolute row index) and its global min / max
// (order-preserving int keys; initialise to INT_MAX / INT_MIN).  map_in: take the values from there instead (function-level
// sw_processing.threshold(img, attention)).
template <int V>
__global__ void __launch_bounds__(ST_THREADS)
stitch_minmax_kernel(const float* __restrict__ lowres, StitchGeom g, const double* __restrict__ wtab, int y_begin, int y_end,
                     int* __restrict__ minmax_ord, float* __restrict__ map_out /*[Ey][Ex] or null*/,
                     const float* __restrict__ map_in /*[Ey][Ex] or null: use instead of stitching lowres*/) {
  __shared__ LinTab tab[ST_MAX_W];
  __shared__ float red_mn[ST_THREADS / 32], red_mx[ST_THREADS / 32];
  if (map_in == nullptr) {
    for (int k = threadIdx.x; k < g.W; k += ST_THREADS) linear_coeff(k, g.scale, g.lw, tab[k].s0, tab[k].s1, tab[k].f);
    __syncthreads();
  }
  const int X0 = st_x0<V>();
  const int dW = g.W / g.S, eW = g.W % g.S;
  float mn = INFINITY, mx = -INFINITY;
  if (X0 < g.Ex) {
    const int q0 = X0 / g.S, r0 = X0 - q0 * g.S;
    for (int Y = y_begin + blockIdx.y; Y < y_end; Y += gridDim.y) {
      float v[V];
      const long long off = static_cast<long long>(Y) * g.Ex + X0;
      if (map_in != nullptr) {
        if (V == 4) {
          const float4 t = *reinterpret_cast<const float4*>(map_in + off);
          v[0] = t.x; v[1 % V] = t.y; v[2 % V] = t.z; v[3 % V] = t.w;
        } else {
          v[0] = map_in[off];
        }
      } else {
        RowCtx rc;
        make_row_ctx(g, Y, rc);
        int q = q0, r = r0;
#pragma unroll
        for (int u = 0; u < V; ++u) {
          v[u] = stitched_value_row(lowres, g, wtab, tab, rc, q, r, dW, eW);
          if (++r == g.S) { r = 0; ++q; }
        }
      }
#pragma unroll
      for (int u = 0; u < V; ++u) { mn = fminf(mn, v[u]); mx = fmaxf(mx, v[u]); }
      if (map_out != nullptr) {
        if (V == 4) *reinterpret_cast<float4*>(map_out + off) = make_float4(v[0], v[1 % V], v[2 % V], v[3 % V]);
        else map_out[off] = v[0];
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < ST_THREADS / 32; ++w) { mn = fminf(mn, red_mn[w]); mx = fmaxf(mx, red_mx[w]); }
    if (mn <= mx) {
      atomicMin(&minmax_ord[0], f2ord(mn));
      atomicMax(&minmax_ord[1], f2ord(mx));
    }
  }
}

// pass 1, column-strip form (the default when the map is stitched from the low-res maps): a thread owns ONE column X over a band
// of SC_ROWS consecutive rows.  Everything that depends on X only (covering tile columns, horizontal bilinear coefficients,
// horizontal blend weights) is computed once per thread; everything that depends on the row only once per row by one thread
// (shared memory); and the horizontal lerps r0 / r1 of bilinear_tab -- which depend on (tile, y0, y1, X) -- stay in registers
// while consecutive rows sample the same pair of low-res rows (8 rows at scale 1/8): per pixel and covering tile that leaves two
// multiplies and an add, plus the fp64 blends.  Same operations in the same order as stitched_value_row (every product and sum
// rounded separately), so the map is bit-identical; the row-organised kernel above needed ~350 instructions per pixel
// (264 us per 4032^2 map), most of them re-deriving these invariants.
constexpr int SC_THREADS = 256;
constexpr int SC_ROWS = 32;
template <int MC>
struct StripRow {
  int ni;                      // covering tile rows
  int base0[MC], base1[MC];    // element offsets of low-res rows y0 / y1 of tile row i0 + k (tile column 0)
  float fy[MC], b0[MC];
  int blend[MC];               // k > 0 && ky < step
  double w[MC], omw[MC];
};
__device__ __forceinline__ float blend_f32_pre(float a, float b, double w, double omw) {   // blend_f32 with 1 - w precomputed
  return static_cast<float>(__dadd_rn(__dmul_rn(static_cast<double>(a), w), __dmul_rn(static_cast<double>(b), omw)));
}
template <int MC>
__global__ void __launch_bounds__(SC_THREADS)
stitch_strip_kernel(const float* __restrict__ lowres, StitchGeom g, const double* __restrict__ wtab, int y_begin, int y_end,
                    int* __restrict__ minmax_ord, float* __restrict__ map_out /*[Ey][Ex] or null*/) {
  __shared__ StripRow<MC> rows[SC_ROWS];
  __shared__ float red_mn[SC_THREADS / 32], red_mx[SC_THREADS / 32];
  const int yb = y_begin + blockIdx.y * SC_ROWS;
  const int nrows = min(SC_ROWS, y_end - yb);
  const int dW = g.W / g.S, eW = g.W % g.S;
  const int lsz = g.lh * g.lw;
  if (static_cast<int>(threadIdx.x) < nrows) {
    const int Y = yb + threadIdx.x;
    StripRow<MC>& R = rows[threadIdx.x];
    const int q = Y / g.S, r = Y - q * g.S;
    int i0, i1;
    cover_range(g.ny, q, r, dW, eW, i0, i1);
    if (i1 - i0 > MC - 1) i1 = i0 + MC - 1;
    R.ni = i1 - i0 + 1;
#pragma unroll
    for (int k = 0; k < MC; ++k) {
      if (k < R.ni) {
        const int i = i0 + k, ky = Y - i * g.S;
        int y0, y1;
        float fy;
        linear_coeff(ky, g.scale, g.lh, y0, y1, fy);
        R.base0[k] = i * g.nx * lsz + y0 * g.lw;
        R.base1[k] = i * g.nx * lsz + y1 * g.lw;
        R.fy[k] = fy;
        R.b0[k] = __fsub_rn(1.0f, fy);
        R.blend[k] = (k > 0 && ky < g.step) ? 1 : 0;
        const double w = R.blend[k] ? wtab[ky] : 0.0;
        R.w[k] = w;
        R.omw[k] = __dsub_rn(1.0, w);
      }
    }
  }
  __syncthreads();
  const int X = blockIdx.x * SC_THREADS + threadIdx.x;
  const bool live = X < g.Ex;
  int nj = 0;
  int o0[MC], o1[MC], bl[MC];
  float fx[MC], a0[MC];
  double wx[MC], omwx[MC];
  if (live) {
    const int q = X / g.S, r = X - q * g.S;
    int j0, j1;
    cover_range(g.nx, q, r, dW, eW, j0, j1);
    if (j1 - j0 > MC - 1) j1 = j0 + MC - 1;
    nj = j1 - j0 + 1;
#pragma unroll
    for (int jj = 0; jj < MC; ++jj) {
      if (jj < nj) {
        const int j = j0 + jj, kx = (q - j) * g.S + r;
        int s0, s1;
        linear_coeff(kx, g.scale, g.lw, s0, s1, fx[jj]);
        a0[jj] = __fsub_rn(1.0f, fx[jj]);
        o0[jj] = j * lsz + s0;
        o1[jj] = j * lsz + s1;
        bl[jj] = (jj > 0 && kx < g.step) ? 1 : 0;
        wx[jj] = bl[jj] ? wtab[kx] : 0.0;
        omwx[jj] = __dsub_rn(1.0, wx[jj]);
      }
    }
  }
  float r0c[MC][MC], r1c[MC][MC];
  int cb0[MC], cb1[MC];
#pragma unroll
  for (int k = 0; k < MC; ++k) { cb0[k] = -1; cb1[k] = -1; }
  float mn = INFINITY, mx = -INFINITY;
  for (int t = 0; t < nrows; ++t) {
    const StripRow<MC>& R = rows[t];
    float v = 0.f;
#pragma unroll
    for (int k = 0; k < MC; ++k) {
      if (k < R.ni) {
        if (R.base0[k] != cb0[k] || R.base1[k] != cb1[k]) {   // (block-uniform) this slot samples other low-res rows than on the previous row
          cb0[k] = R.base0[k];
          cb1[k] = R.base1[k];
          const float* p0 = lowres + cb0[k];
          const float* p1 = lowres + cb1[k];
#pragma unroll
          for (int jj = 0; jj < MC; ++jj) {
            if (jj < nj) {
              r0c[k][jj] = __fadd_rn(__fmul_rn(__ldg(p0 + o0[jj]), a0[jj]), __fmul_rn(__ldg(p0 + o1[jj]), fx[jj]));
              r1c[k][jj] = __fadd_rn(__fmul_rn(__ldg(p1 + o0[jj]), a0[jj]), __fmul_rn(__ldg(p1 + o1[jj]), fx[jj]));
            }
          }
        }
        float hv = 0.f;
#pragma unroll
        for (int jj = 0; jj < MC; ++jj) {
          if (jj < nj) {
            const float tv = __fadd_rn(__fmul_rn(r0c[k][jj], R.b0[k]), __fmul_rn(r1c[k][jj], R.fy[k]));
            hv = bl[jj] ? blend_f32_pre(hv, tv, wx[jj], omwx[jj]) : tv;
          }
        }
        v = R.blend[k] ? blend_f32_pre(v, hv, R.w[k], R.omw[k]) : hv;
      }
    }
    if (live) {
      mn = fminf(mn, v);
      mx = fmaxf(mx, v);
      if (map_out != nullptr) map_out[static_cast<long long>(yb + t) * g.Ex + X] = v;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) { red_mn[threadIdx.x >> 5] = mn; red_mx[threadIdx.x >> 5] = mx; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < SC_THREADS / 32; ++w) { mn = fminf(mn, red_mn[w]); mx = fmaxf(mx, red_mx[w]); }
    if (mn <= mx) {
      atomicMin(&minmax_ord[0], f2ord(mn));
      atomicMax(&minmax_ord[1], f2ord(mx));
    }
  }
}

// per-pixel classification of the mosaic flavour (SSS/sw_processing.py:43-48)
__device__ __forceinline__ void sw_classify(float v, float mn, float range, bool flat, float att_max, int img, int& res, int& au) {
  const float an = flat ? v : __fdiv_rn(__fsub_rn(v, mn), range);
  res = static_cast<int>(static_cast<uint8_t>(static_cast<int>(__fdiv_rn(__fmul_rn(static_cast<float>(img), an), att_max))));
  au = static_cast<int>(static_cast<uint8_t>(static_cast<int>(__fmul_rn(an, 255.0f))));
}

// V stitched values + V gray bytes of (Y, X0 ...): the map comes from map_in when given (the fast path: pass 1 stored it),
// else it is re-evaluated from the low-res maps
template <int V>
__device__ __forceinline__ void st_load_px(const float* __restrict__ lowres, const StitchGeom& g, const double* __restrict__ wtab,
                                           const LinTab* __restrict__ tab, const float* __restrict__ map_in, const uint8_t* __restrict__ gray,
                                           int Y, int X0, int q0, int r0, float (&v)[V], int (&img)[V]) {
  const long long off = static_cast<long long>(Y) * g.Ex + X0;
  if (map_in != nullptr) {
    if (V == 4) {
      const float4 t = *reinterpret_cast<const float4*>(map_in + off);
      v[0] = t.x; v[1 % V] = t.y; v[2 % V] = t.z; v[3 % V] = t.w;
    } else {
      v[0] = map_in[off];
    }
  } else {
    RowCtx rc;
    make_row_ctx(g, Y, rc);
    int q = q0, r = r0;
    const int dW = g.W / g.S, eW = g.W % g.S;
#pragma unroll
    for (int u = 0; u < V; ++u) {
      v[u] = stitched_value_row(lowres, g, wtab, tab, rc, q, r, dW, eW);
      if (++r == g.S) { r = 0; ++q; }
    }
  }
  if (V == 4) {
    const uchar4 b = *reinterpret_cast<const uchar4*>(gray + off);
    img[0] = b.x; img[1 % V] = b.y; img[2 % V] = b.z; img[3 % V] = b.w;
  } else {
    img[0] = gray[off];
  }
}

// pass 2: histograms of result (= img * att), of the stitched gray image and of att_u8 -> hists[3][256].
// One private histogram set per warp (the images are dark: a block-wide table serialises on a few bins).
template <int V>
__global__ void __launch_bounds__(ST_THREADS)
stitch_hist_kernel(const float* __restrict__ lowres, StitchGeom g, const double* __restrict__ wtab,
                   const uint8_t* __restrict__ gray /*[Ey][Ex]*/, const int* __restrict__ minmax_ord, int y_begin, int y_end,
                   unsigned long long* __restrict__ hists, const float* __restrict__ map_in) {
  __shared__ LinTab tab[ST_MAX_W];
  __shared__ unsigned int h[ST_THREADS / 32][3][256];
  for (int i = threadIdx.x; i < (ST_THREADS / 32) * 3 * 256; i += ST_THREADS) (&h[0][0][0])[i] = 0u;
  if (map_in == nullptr)
    for (int k = threadIdx.x; k < g.W; k += ST_THREADS) linear_coeff(k, g.scale, g.lw, tab[k].s0, tab[k].s1, tab[k].f);
  __syncthreads();
  const float mn = ord2f(minmax_ord[0]), mx = ord2f(minmax_ord[1]);
  const bool flat = (mx == mn);
  const float range = __fsub_rn(mx, mn);
  const float att_max = flat ? mx : 1.0f;  // np.max(attention) after min_max_normalize
  const int X0 = st_x0<V>();
  unsigned int (*hw)[256] = h[threadIdx.x >> 5];
  if (X0 < g.Ex) {
    const int q0 = X0 / g.S, r0 = X0 - q0 * g.S;
    for (int Y = y_begin + blockIdx.y; Y < y_end; Y += gridDim.y) {
      float v[V];
      int img[V];
      st_load_px<V>(lowres, g, wtab, tab, map_in, gray, Y, X0, q0, r0, v, img);
#pragma unroll
      for (int u = 0; u < V; ++u) {
        int res, au;
        sw_classify(v[u], mn, range, flat, att_max, img[u], res, au);
        atomicAdd(&hw[0][res], 1u);
        atomicAdd(&hw[1][img[u]], 1u);
        atomicAdd(&hw[2][au], 1u);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * 256; i += ST_THREADS) {
    unsigned int c = 0;
#pragma unroll
    for (int w = 0; w < ST_THREADS / 32; ++w) c += (&h[w][0][0])[i];
    if (c) atomicAdd(&hists[i], static_cast<unsigned long long>(c));
  }
}

// pass 3: masks th (result > t0), th2 (gray > t1), th3 (att_u8 > t2); rows [y_begin, y_end) written at
// out + (Y - y_begin) * Ex so that a rank can hold only its own band.
template <int V>
__global__ void __launch_bounds__(ST_THREADS)
stitch_mask_kernel(const float* __restrict__ lowres, StitchGeom g, const double* __restrict__ wtab,
                   const uint8_t* __restrict__ gray, const int* __restrict__ minmax_ord, const int* __restrict__ thr,
                   int y_begin, int y_end, uint8_t* __restrict__ th, uint8_t* __restrict__ th2, uint8_t* __restrict__ th3,
                   const float* __restrict__ map_in) {
  __shared__ LinTab tab[ST_MAX_W];
  if (map_in == nullptr) {
    for (int k = threadIdx.x; k < g.W; k += ST_THREADS) linear_coeff(k, g.scale, g.lw, tab[k].s0, tab[k].s1, tab[k].f);
    __syncthreads();
  }
  const float mn = ord2f(minmax_ord[0]), mx = ord2f(minmax_ord[1]);
  const bool flat = (mx == mn);
  const float range = __fsub_rn(mx, mn);
  const float att_max = flat ? mx : 1.0f;
  const int t0 = thr[0], t1 = thr[1], t2 = thr[2];
  const int X0 = st_x0<V>();
  if (X0 >= g.Ex) return;
  const int q0 = X0 / g.S, r0 = X0 - q0 * g.S;
  for (int Y = y_begin + blockIdx.y; Y < y_end; Y += gridDim.y) {
    float v[V];
    int img[V];
    st_load_px<V>(lowres, g, wtab, tab, map_in, gray, Y, X0, q0, r0, v, img);
    uint8_t m0[V], m1[V], m2[V];
#pragma unroll
    for (int u = 0; u < V; ++u) {
      int res, au;
      sw_classify(v[u], mn, range, flat, att_max, img[u], res, au);
      m0[u] = res > t0 ? 255 : 0;
      m1[u] = img[u] > t1 ? 255 : 0;
      m2[u] = au > t2 ? 255 : 0;
    }
    const long long o = static_cast<long long>(Y - y_begin) * g.Ex + X0;
    if (V == 4) {
      if (th != nullptr) *reinterpret_cast<uchar4*>(th + o) = make_uchar4(m0[0], m0[1 % V], m0[2 % V], m0[3 % V]);
      if (th2 != nullptr) *reinterpret_cast<uchar4*>(th2 + o) = make_uchar4(m1[0], m1[1 % V], m1[2 % V], m1[3 % V]);
      if (th3 != nullptr) *reinterpret_cast<uchar4*>(th3 + o) = make_uchar4(m2[0], m2[1 % V], m2[2 % V], m2[3 % V]);
    } else {
      if (th != nullptr) th[o] = m0[0];
      if (th2 != nullptr) th2[o] = m1[0];
      if (th3 != nullptr) th3[o] = m2[0];
    }
  }
}

// the weighted image `result = (img * att / max(att)).astype(u8)` of the mosaic flavour (SSS/sw_processing.py:44-46, the
// "weighted_iamge_attention.png" it saves at :75) and att_u8, for rows [y_begin, y_end)
template <int V>
__global__ void __launch_bounds__(ST_THREADS)
stitch_result_kernel(const float* __restrict__ lowres, StitchGeom g, const double* __restrict__ wtab, const uint8_t* __restrict__ gray,
                     const int* __restrict__ minmax_ord, int y_begin, int y_end, uint8_t* __restrict__ result, uint8_t* __restrict__ att_u8,
                     const float* __restrict__ map_in) {
  __shared__ LinTab tab[ST_MAX_W];
  if (map_in == nullptr) {
    for (int k = threadIdx.x; k < g.W; k += ST_THREADS) linear_coeff(k, g.scale, g.lw, tab[k].s0, tab[k].s1, tab[k].f);
    __syncthreads();
  }
  const float mn = ord2f(minmax_ord[0]), mx = ord2f(minmax_ord[1]);
  const bool flat = (mx == mn);
  const float range = __fsub_rn(mx, mn);
  const float att_max = flat ? mx : 1.0f;
  const int X0 = st_x0<V>();
  if (X0 >= g.Ex) return;
  const int q0 = X0 / g.S, r0 = X0 - q0 * g.S;
  for (int Y = y_begin + blockIdx.y; Y < y_end; Y += gridDim.y) {
    float v[V];
    int img[V];
    st_load_px<V>(lowres, g, wtab, tab, map_in, gray, Y, X0, q0, r0, v, img);
    const long long o = static_cast<long long>(Y - y_begin) * g.Ex + X0;
#pragma unroll
    for (int u = 0; u < V; ++u) {
      int res, au;
      sw_classify(v[u], mn, range, flat, att_max, img[u], res, au);
      if (result != nullptr) result[o + u] = static_cast<uint8_t>(res);
      if (att_u8 != nullptr) att_u8[o + u] = static_cast<uint8_t>(au);
    }
  }
}

}  // namespace vitocm
