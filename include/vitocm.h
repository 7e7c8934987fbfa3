/* vitocm.h -- C ABI of libvitocm.so, the B200 (sm_100a) implementation of the ViT-OCM
 * attention-map / sliding-window segmentation hot path.
 *
 * The reference (linum-uqam/ViT-OCM-WMSegmentation) has NO FFI, plugin or operator interface:
 * its boundary for this path is the Python nn.Module surface of
 * Self-supervised_segmentation/dino/vision_transformer.py (abbrev. vit.py) plus a handful of
 * post-processing functions (SURVEY.md section 8b).  Each entry point below therefore cites
 * the reference Python function(s) whose arithmetic it replaces; the Python mirror of that
 * surface (same class / function names and arguments) lives in vit-ocm-wmsegmentation_b200/
 * and binds these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions: every function returns 0 on success or a negative vitocm_status; the message of
 * the last failure on the calling thread is vitocm_last_error().  No exception crosses the
 * ABI.  All data pointers are DEVICE pointers unless the parameter is named host_*; tensors
 * are dense row-major.  `stream` is a cudaStream_t passed as void*.  No hidden device
 * allocation on the forward paths: the caller passes a workspace sized by
 * vitocm_workspace_bytes().  A handle is thread-compatible (one thread at a time).
 */
#ifndef VITOCM_H_
#define VITOCM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VITOCM_VERSION 100

typedef enum vitocm_status {
  VITOCM_OK = 0,
  VITOCM_ERR_INVALID = -1,   /* bad argument / unsupported shape */
  VITOCM_ERR_CUDA = -2,      /* CUDA runtime or driver error */
  VITOCM_ERR_STATE = -3,     /* weights missing / not finalized */
  VITOCM_ERR_WORKSPACE = -4  /* workspace too small */
} vitocm_status;

typedef enum vitocm_precision {
  VITOCM_BF16 = 0, /* bf16 tensor-core operands, fp32 accumulate / residual / LN / softmax statistics */
  VITOCM_FP32 = 1, /* fp32-parity mode: every operand a bf16 (hi, lo) pair, products hi*hi+hi*lo+lo*hi */
  VITOCM_FP16 = 2  /* IEEE fp16 tensor-core operands (11 significand bits instead of 8, same rate), saturating conversions,
                    * fp32 accumulate / residual / LN / softmax statistics: the inference default -- the reference is an fp32
                    * model (vit.py:78-90, no autocast anywhere) and its masks need ~1e-4 relative CLS rows (DESIGN.md 4) */
} vitocm_precision;

/* Constructor constants of VisionTransformer (vit.py:137-139) and of the factories
 * vit_tiny/small/base (vit.py:259-279).  head_dim = embed_dim / num_heads must be 64 or 128. */
typedef struct vitocm_config {
  int embed_dim;
  int depth;
  int num_heads;
  int mlp_hidden;
  int patch_size;
  int in_chans;
  float ln_eps;
  float qk_scale; /* head_dim ** -0.5 unless qk_scale was given (vit.py:70-71) */
  int precision;  /* vitocm_precision */
} vitocm_config;

typedef struct vitocm_engine vitocm_engine;

int vitocm_version(void);
const char* vitocm_last_error(void);

int vitocm_create(const vitocm_config* cfg, vitocm_engine** out);
int vitocm_destroy(vitocm_engine* e);

/* Replaces nn.Module.load_state_dict for the hot path (SSS/eval.py:67-77): `name` is a
 * state-dict key (cls_token, pos_embed, mask_token, decoder.0.{weight,bias} (MIM), patch_embed.proj.{weight,bias},
 * blocks.{i}.{norm1,norm2}.{weight,bias}, blocks.{i}.attn.{qkv,proj}.{weight,bias},
 * blocks.{i}.mlp.{fc1,fc2}.{weight,bias}, norm.{weight,bias}); host_data is fp32, `numel`
 * elements.  vitocm_finalize_weights repacks them into the kernels' layouts (bf16 hi/lo,
 * transposed patch filter) and must be called after the last load and before any forward.  For single 16-bit engines at
 * embed_dim 128 / 384 it also folds the LayerNorm affine parameters into the Linear behind them (fc1 <- norm2, qkv <- norm1:
 * W' = W diag(gamma), b' = b + W beta, from the fp32 masters) for the block-tail kernel; vitocm_refresh_weights drops those copies
 * (the forward then applies gamma / beta itself) until the next vitocm_finalize_weights.  VITOCM_TAIL_FOLD=0 (read at
 * vitocm_create) disables the folding. */
int vitocm_load_weight(vitocm_engine* e, const char* name, const float* host_data, int64_t numel);
int vitocm_finalize_weights(vitocm_engine* e);

/* Precision schedule, per transformer block (call before vitocm_workspace_bytes / the forwards; bf16 and fp16 engines):
 * mode 0 = the engine's precision; mode 1 = this block's fc1 / fc2 (vit.py:57-63) read their activations -- norm2's output and
 * gelu(fc1) -- as (hi, lo) pairs of the engine's 16-bit format against single-precision weights, two MMAs per product.  These two
 * roundings carry ~70 % of the CLS-row error variance of a 16-bit forward (profiles/r02_precision_sim.txt). */
int vitocm_set_layer_mode(vitocm_engine* e, int layer, int mode);

/* Bytes of workspace needed by the forward entry points for chunks of `chunk_tiles` images of
 * n_tokens tokens each. */
size_t vitocm_workspace_bytes(const vitocm_engine* e, int chunk_tiles, int n_tokens);

/* Chunk-level concurrency of vitocm_forward_cls_attn: `lanes` (1..4) independent chunks of tiles are processed
 * concurrently, lane 0 on the caller's stream, the others on streams owned by the engine (forked from / joined back
 * into the caller's stream with events).  vitocm_workspace_bytes accounts for the configured number of lanes. */
int vitocm_set_concurrency(vitocm_engine* e, int lanes);

/* HOT PATH.  VisionTransformer.get_last_selfattention(x)[:, :, 0, :] (vit.py:239-246), i.e. the
 * CLS query row per head that SSS/utils.py:232 (query = 0) slices out of
 * get_intermediate_feat(x, n=1) (vit.py:225-237; callers SSS/eval.py:136, SSS/sw_processing.py:239).
 * x [B][C][H][W] fp32; pos [1 + (H/p)(W/p)][D] fp32 = (interpolated) position table (vit.py:176-196);
 * out_rows [B][heads][N] fp32.  Internally: patch embedding, depth-1 full blocks, and for the last
 * block only LN1 -> K projection -> softmax(q_cls K^T).  Processes the batch in chunks that fit ws. */
int vitocm_forward_cls_attn(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, float* out_rows,
                            void* ws, size_t ws_bytes, int chunk_tiles, void* stream);

/* Images of different sizes in one forward (the reference runs each image at its own size: SSS/eval.py:126-136,
 * SSS/analyse_attention.py:113-177; its datasets only crop to a multiple of 8, SSS/data.py:29-30).  B images packed back to back in
 * x as fp32 [C][H_i][W_i] (C = in_chans, or 1 for the gray channel-folded path of vitocm_forward_cls_attn_gray); hw host int
 * [B][2] = (H_i, W_i), positive multiples of the patch size; N_i = (H_i/p)(W_i/p) + 1.  pos: the packed position tables, one per
 * distinct size (each [N][D] fp32 as in vitocm_forward_cls_attn); pos_off host int [B]: image i's table starts at row pos_off[i].
 * out_rows fp32: image i owns the [heads][N_i] block at heads * sum_{j<i} N_j.  The token rows of all images form one stream
 * through every kernel that works on rows; patch embedding, attention and the CLS row take per-image geometry from tables the call
 * writes into ws on `stream` (nothing allocated on the device).  Images are taken in order into chunks of at most
 * chunk_tokens rows (<= 0: VITOCM_VARLEN_CHUNK_TOKENS); an image of more tokens than that runs alone.  One lane: the chunks run
 * on `stream` one after the other (vitocm_set_concurrency does not apply).  Each image's rows are bit-identical to
 * vitocm_forward_cls_attn(_gray) of that image alone on the same engine.  Refused: B < 1, a size that is not a multiple of the
 * patch, an N_i whose CLS row does not fit the CLS-row kernel's shared memory, a workspace below
 * vitocm_varlen_workspace_bytes(e, T) with T = the tokens of the largest chunk (at most max(chunk_tokens, largest N_i) and at most
 * sum N_i).  The tables go to the device from pinned memory owned by the engine, in two slots used by calls in turn: a call waits on
 * the host only for the table copies of the call before the previous one. */
#define VITOCM_VARLEN_CHUNK_TOKENS 401920 /* 512 images of 224^2 at patch 8 */
size_t vitocm_varlen_workspace_bytes(const vitocm_engine* e, int64_t chunk_tokens);
int vitocm_forward_cls_attn_varlen(vitocm_engine* e, const float* x, int B, int C, const int* hw, const float* pos, const int* pos_off,
                                   float* out_rows, void* ws, size_t ws_bytes, int64_t chunk_tokens, void* stream);

/* Gray fast path of vitocm_forward_cls_attn: x [B][1][H][W] fp32 stands for an image whose in_chans channels are all equal
 * (every OCM tile of the reference: PIL "RGB" of a gray PNG, SSS/sw_processing.py:225-236).  The patch filter is folded over
 * the channels at vitocm_finalize_weights, so the patch-embedding GEMM contracts over p*p instead of in_chans*p*p taps and the
 * tiles are a third of the bytes; same arithmetic up to fp32 summation order. */
int vitocm_forward_cls_attn_gray(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, float* out_rows,
                                 void* ws, size_t ws_bytes, int chunk_tiles, void* stream);
/* The same with the tiles cut straight out of a gray uint8 mosaic by the patch-embedding producer -- sliding_window + ToTensor
 * (SSS/sw_processing.py:151-163, :236) without materialised crops: tile t0 + i (i < T) is the W x W window of the n x n grid at
 * stride S, origin ((t / n) * S, (t % n) * S), pixel value v / 255, zero beyond the mosaic (PIL's crop).  mosaic [mos_h][pitch]
 * device memory; out_rows [T][heads][N]. */
int vitocm_forward_cls_attn_mosaic(vitocm_engine* e, const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int n, int W, int S,
                                   int t0, int T, const float* pos, float* out_rows, void* ws, size_t ws_bytes, int chunk_tiles,
                                   void* stream);
/* The same on a rectangular ny x nx grid (rows of windows over the mosaic's height, columns over its width; the reference's
 * SSS/sw_processing.py:151-163 walk with the axes taken from the height and the width of a rectangle): window t0 + i has origin
 * ((t / nx) * S, (t % nx) * S).  Needs ny, nx >= 1 and t0 + T <= ny * nx.  vitocm_forward_cls_attn_mosaic is this with ny = nx = n. */
int vitocm_forward_cls_attn_mosaic_grid(vitocm_engine* e, const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int ny, int nx, int W,
                                        int S, int t0, int T, const float* pos, float* out_rows, void* ws, size_t ws_bytes, int chunk_tiles,
                                        void* stream);

/* The same forward for a LIST of query tokens (SSS/analyse_attention.py:183-247: compute_attention(..., query=q) for a
 * region query) and, optionally, the last block's K features (SSS/analyse_attention.py:139-163, SSS/eval.py:186-202, the
 * input of the k-means feature clustering): queries = DEVICE int32 [nq] token indices in [0, N) (0 = CLS, 1 + i = patch i);
 * out_rows [B][heads][nq][N] fp32 = get_last_selfattention(x)[:, :, queries, :]; k_out [B][N][D] fp32 (K projection of the
 * last block including its bias, heads side by side = qkv[1] of vit.py:81 before the head split) or NULL. */
int vitocm_forward_query_attn(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const int* queries, int nq,
                              float* out_rows, float* k_out, void* ws, size_t ws_bytes, int chunk_tiles, void* stream);

/* prepare_tokens (vit.py:198-209): patch embedding + CLS + position add -> X [B][N][D] fp32.
 * mask [B][n] fp32 in {0,1} or NULL: SimMIM mask-token mixing (SSS/model.py:31-33). */
int vitocm_prepare_tokens(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask,
                          float* X, void* stream);

/* Block.forward (vit.py:106-114) in place on X [B][N][D] fp32 for block index `layer`. */
int vitocm_block_forward(vitocm_engine* e, int layer, float* X, int B, int n_tokens, void* ws, size_t ws_bytes,
                         void* stream);

/* Attention probabilities of block `layer` for input X (vit.py:78-84, the `attn` that
 * Block.forward(return_attention=True) returns): attn [B][heads][N][N] fp32; qkv_out
 * [B*N][3D] fp32 (the pre-permute qkv activation, vit.py:80) -- required scratch/output. */
int vitocm_block_attn_probs(vitocm_engine* e, int layer, const float* X, int B, int n_tokens, float* attn,
                            float* qkv_out, void* ws, size_t ws_bytes, void* stream);

/* MIM.forward (SSS/model.py:71-77) without autograd: VisionTransformerForSimMIM.forward (model.py:25-53: patch embed,
 * mask-token mixing, cls, pos, all blocks, norm) -> 1x1-conv decoder + PixelShuffle(patch) (model.py:61-66) -> masked L1.
 * Needs the weights "mask_token", "decoder.0.weight" [C p^2][D] and "decoder.0.bias".  x [B][C][H][W]; mask [B][n] fp32
 * in {0,1} (MaskGenerator, SSS/data.py:163-186); x_rec [B][C][H][W] fp32; loss_sums double[2] = {sum |x - x_rec| * mask,
 * sum mask}: loss = loss_sums[0] / (loss_sums[1] + 1e-5) / C (model.py:75-76). */
int vitocm_mim_forward(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask, float* x_rec,
                       double* loss_sums, void* ws, size_t ws_bytes, int chunk_tiles, void* stream);

/* self.norm (vit.py:215, :234): out [M][D] fp32 = LayerNorm(X [M][D]). */
int vitocm_final_norm(vitocm_engine* e, const float* X, float* out, int M, void* stream);

/* ---- post-processing (SSS/utils.py, SSS/eval.py, SSS/sw_processing.py) ---- */

/* rows [T][heads][N] -> lowres [T][N-1]: head mean of the CLS row without its CLS column
 * (SSS/utils.py:232-233 + np.mean at SSS/eval.py:142).  mode 1 also applies the per-tile
 * (a-min)/(max-min)*255 of SSS/sw_processing.py:253-254. */
int vitocm_head_mean(const float* rows, float* lowres, int T, int heads, int n_tokens, int mode, void* stream);

/* vitocm_head_mean for T images of different sizes packed as vitocm_forward_cls_attn_varlen writes them: patch_off device int [T + 1]
 * = patches before image t (patch_off[T] = all); image t's rows are [heads][N_t] at heads (patch_off[t] + t), N_t = patch_off[t + 1]
 * - patch_off[t] + 1, and its map lowres[patch_off[t] ...] [h_t][w_t]. */
int vitocm_head_mean_varlen(const float* rows, float* lowres, int T, int heads, const int* patch_off, int mode, void* stream);

/* Cumulative-mass threshold per head (the `--threshold` flag whose help text is at SSS/eval.py:33-34; the arithmetic is upstream
 * DINO's visualize_attention.py, not under /root/reference: parity unpinned by the reference, oracle = a PyTorch restatement):
 * per (tile, head) over the N - 1 patch columns of the CLS row: sort ascending, normalise by the sum, cumulative sum, keep the
 * patches whose cumulative mass exceeds 1 - threshold, back in patch order.  rows [T][heads][N] fp32 -> mask [T][heads][N-1] u8
 * in {0,1}; up [T][heads][lh*patch][lw*patch] fp32 (optional, NULL to skip) = the nearest x patch upsampling of the mask. */
int vitocm_attn_cummass(const float* rows, int T, int heads, int n_tokens, float threshold, uint8_t* mask, float* up, int lh, int lw,
                        int patch, void* stream);

/* SSS/eval.py:169-173 + utils.threshold (SSS/utils.py:62-115) for T images: lowres [T][lh][lw],
 * x [T][C][S][S] fp32 in [0,1]; masks [T][3][S][S] u8 = (th "ours", th2 "otsu", th3 "heatmap_threshold");
 * thresholds [T][3] int32; att_out [T][S][S] fp32 or NULL (the bilinearly upsampled map).
 * att_in [T][S][S] fp32 (optional): a caller-supplied full-resolution attention map, used instead of
 * upsampling lowres -- this is the exact signature of utils.threshold(img, attention).
 * img_in [T][S][S] u8 (optional): the PIL "L" image, used instead of deriving it from x. */
int vitocm_tile_threshold(const float* lowres, const float* x, int T, int C, int S, int lh, int lw, uint8_t* masks,
                          int* thresholds, float* att_out, const float* att_in, const uint8_t* img_in, void* stream);
/* vitocm_tile_threshold for T square images of different sides: geo device int [T][4] = (S_t, l_t, patch offset, pixel offset):
 * lowres [l_t][l_t] at the patch offset (vitocm_head_mean_varlen's layout), x [C][S_t][S_t] at C x the pixel offset, masks
 * [3][S_t][S_t] at 3 x it and att_out [S_t][S_t] (or NULL) at it; thresholds [T][3]. */
int vitocm_tile_threshold_varlen(const float* lowres, const float* x, int T, int C, const int* geo, uint8_t* masks, int* thresholds,
                                 float* att_out, void* stream);
/* The same with the two images utils.threshold also writes out (SSS/utils.py:77-81, saved at :107-108): aux [T][2][S][S] u8 =
 * (result = the 0.6 / 0.4 image / attention blend "weighted_iamge_attention.png", att_u8 = the normalised attention * 255). */
int vitocm_tile_threshold_aux(const float* lowres, const float* x, int T, int C, int S, int lh, int lw, uint8_t* masks,
                              int* thresholds, float* att_out, const float* att_in, const uint8_t* img_in, uint8_t* aux, void* stream);

/* sliding_window (SSS/sw_processing.py:151-163) + ToTensor for tiles t0..t0+T-1 of an n x n grid:
 * mosaic u8 gray [mos_h][pitch] -> x [T][C][W][W] fp32. */
int vitocm_extract_tiles(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int n, int W, int S, int t0, int T,
                         int C, float* x, void* stream);
/* The same for tiles t0..t0+T-1 (row-major) of an ny x nx grid (SSS/sw_processing.py:151-163 with rows over the height and
 * columns over the width); needs t0 + T <= ny * nx. */
int vitocm_extract_tiles_grid(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int ny, int nx, int W, int S, int t0, int T,
                              int C, float* x, void* stream);

/* concat_crops on the uint8 image crops (SSS/sw_processing.py:113-149 at :225) for output rows
 * [y_begin, y_end): out [E][E] u8 (full-size buffer, E = (n-1) S + W).  wtab = host-computed
 * numpy.linspace(1, 0, W - S) copied to the device (double[W - S]). */
int vitocm_stitch_gray(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int n, int W, int S,
                       const double* wtab, int y_begin, int y_end, uint8_t* out, void* stream);

/* Rectangular grids.  The *_grid forms below take an ny x nx window grid where the functions above take n (each n-form is its
 * grid form with ny = nx = n): tile t = i * nx + j sits at (i S, j S); the stitched extent is Ey x Ex = ((ny-1) S + W) x
 * ((nx-1) S + W); concat_crops (SSS/sw_processing.py:113-134) blends along x inside each of the ny strips of nx crops, then along
 * y across the strips, in the reference's order with its ramp and its truncations.  Row bands [y_begin, y_end) lie in [0, Ey);
 * full-size buffers (gray, map_out, map_in) have row pitch Ex; per-band outputs are [(y_end-y_begin)][Ex].  With map_in and
 * lowres == NULL only the extent of the geometry is used: any (ny, nx, W, S) whose extent is the map's addresses it (e.g.
 * W = 2, S = 1, ny = Ey - 1, nx = Ex - 1).  Grids with ny, nx < 1, W <= S or W > 4 S, and bands outside [0, Ey) are refused
 * before any launch. */
int vitocm_stitch_gray_grid(const uint8_t* mosaic, int mos_h, int mos_w, int64_t pitch, int ny, int nx, int W, int S,
                            const double* wtab, int y_begin, int y_end, uint8_t* out, void* stream);

/* Stitched attention map = resize pair (SSS/sw_processing.py:255-257) + concat_crops (:259) of the
 * per-tile maps lowres [n*n][lh][lw]; pass 1 of sw_processing.threshold (:43): global min / max over
 * rows [y_begin, y_end) accumulated into minmax_ord[2] (order-preserving int keys; initialise with
 * vitocm_minmax_init).  map_out [E][E] fp32 or NULL.  map_in [E][E] fp32 (optional, also on the two
 * passes below): a caller-supplied stitched map used instead of stitching lowres -- the exact
 * signature of sw_processing.threshold(img, attention). */
int vitocm_minmax_init(int* minmax_ord, void* stream);
int vitocm_stitch_minmax(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab, int y_begin,
                         int y_end, int* minmax_ord, float* map_out, const float* map_in, void* stream);

/* pass 2 (SSS/sw_processing.py:44-48): 256-bin histograms of result = u8(img*att), of the stitched
 * gray image and of att_u8, accumulated into hists[3][256] (uint64; caller zeroes). */
int vitocm_stitch_hist(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab,
                       const uint8_t* gray, const int* minmax_ord, int y_begin, int y_end, uint64_t* hists,
                       const float* map_in, void* stream);

/* cv2.threshold(..., THRESH_OTSU) threshold selection for nhist histograms [nhist][256] uint64. */
int vitocm_otsu(const uint64_t* hists, int nhist, int* thresholds, void* stream);

/* pass 3 (SSS/sw_processing.py:54-61): masks for rows [y_begin, y_end), each [(y_end-y_begin)][E] u8
 * (any may be NULL): th = result > thr[0], th2 = gray > thr[1], th3 = att_u8 > thr[2]. */
int vitocm_stitch_mask(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab,
                       const uint8_t* gray, const int* minmax_ord, const int* thr, int y_begin, int y_end, uint8_t* th,
                       uint8_t* th2, uint8_t* th3, const float* map_in, void* stream);

/* The weighted image of the mosaic flavour, result = (img * att / max(att)).astype(u8) (SSS/sw_processing.py:44-46, saved as
 * "weighted_iamge_attention.png" at :75), and att_u8 (:47-48) for rows [y_begin, y_end): each [(y_end-y_begin)][E] u8 or NULL. */
int vitocm_stitch_result(const float* lowres, int n, int W, int S, int lh, int lw, const double* wtab, const uint8_t* gray,
                         const int* minmax_ord, int y_begin, int y_end, uint8_t* result, uint8_t* att_u8, const float* map_in,
                         void* stream);

/* Grid forms of the three passes and of the weighted image (SSS/sw_processing.py:37-61, :255-259 on an ny x nx grid; see
 * vitocm_stitch_gray_grid for the geometry): lowres [ny*nx][lh][lw] row-major; map_in / map_out [Ey][Ex]. */
int vitocm_stitch_minmax_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab, int y_begin,
                              int y_end, int* minmax_ord, float* map_out, const float* map_in, void* stream);
int vitocm_stitch_hist_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab,
                            const uint8_t* gray, const int* minmax_ord, int y_begin, int y_end, uint64_t* hists,
                            const float* map_in, void* stream);
int vitocm_stitch_mask_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab,
                            const uint8_t* gray, const int* minmax_ord, const int* thr, int y_begin, int y_end, uint8_t* th,
                            uint8_t* th2, uint8_t* th3, const float* map_in, void* stream);
int vitocm_stitch_result_grid(const float* lowres, int ny, int nx, int W, int S, int lh, int lw, const double* wtab,
                              const uint8_t* gray, const int* minmax_ord, int y_begin, int y_end, uint8_t* result, uint8_t* att_u8,
                              const float* map_in, void* stream);

/* concat_crops(crops, stride, window_size) (SSS/sw_processing.py:113-149) on full-resolution crops:
 * float32 [n*n][W][W] -> out [E][E]; uint8 HWC [n*n][W][W][C] -> out [E][E][C]. */
int vitocm_concat_crops_f32(const float* crops, int n, int W, int S, const double* wtab, float* out, void* stream);
int vitocm_concat_crops_u8(const uint8_t* crops, int n, int W, int S, int C, const double* wtab, uint8_t* out,
                           void* stream);
/* The same on a row-major ny x nx grid of crops (SSS/sw_processing.py:113-134 with the strip loop over ny and the crop loop
 * over nx): float32 [ny*nx][W][W] -> out [Ey][Ex]; uint8 HWC [ny*nx][W][W][C] -> out [Ey][Ex][C]. */
int vitocm_concat_crops_grid_f32(const float* crops, int ny, int nx, int W, int S, const double* wtab, float* out, void* stream);
int vitocm_concat_crops_grid_u8(const uint8_t* crops, int ny, int nx, int W, int S, int C, const double* wtab, uint8_t* out,
                                void* stream);
/* sliding_window(image, stride, window_size) (SSS/sw_processing.py:151-163) on a uint8 HWC image:
 * ny x nx windows at stride S -> crops [ny*nx][W][W][C], zero padded outside the image. */
int vitocm_crop_u8(const uint8_t* img, int img_h, int img_w, int C, int ny, int nx, int W, int S, uint8_t* crops,
                   void* stream);

/* concat_crops_overlap(crops, stride) (SSS/utils.py:319-347): n x n crops of size W overlapping by 2*stride,
 * overlaps = floor-halved sum `a // 2 + b // 2` along x then along y; the last strip is appended unblended
 * (:337-339).  float32 [n*n][W][W] -> out [E][E]; uint8 HWC [n*n][W][W][C] -> out [E][E][C];
 * E = W + (n-1) * (W - 2*stride).  Needs 0 < 2*stride < W. */
int vitocm_concat_crops_overlap_f32(const float* crops, int n, int W, int stride, float* out, void* stream);
int vitocm_concat_crops_overlap_u8(const uint8_t* crops, int n, int W, int stride, int C, uint8_t* out, void* stream);
/* Plain tiling `concat_crops(crops)` (SSS/utils.py:304-317) of channel c0 of batched crops, as the `--crop 4|16`
 * evaluation does for the attention maps and the image (SSS/eval.py:160-161):
 * src [B][cr*cr][C][h][w] fp32 -> dst [B][cr*h][cr*w]. */
int vitocm_concat_grid_f32(const float* src, int B, int cr, int C, int c0, int h, int w, float* dst, void* stream);

/* ---- kernel-level entry points used by the tests / the bench roofline leg ---- */

/* C = epilogue(A[M][K] . B[N][K]^T): A, B bf16 device (split: [rows][2K] = hi|lo); epilogue enum:
 * 0 bias->bf16, 1 bias+gelu->bf16, 2 bias + in-place fp32 residual add, 3 bias->fp32.
 * split_out (16-bit outputs): 1 = out[:, lo_off:lo_off+N] also receives lo = v - 16-bit(v); 2 with epilogue 1 (the training fc1) =
 * out[:, :N] = gelu(pre) and out[:, lo_off:lo_off+N] = pre = acc + bias, the GELU input the backward reads. */
int vitocm_gemm(vitocm_engine* e, const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K,
                int split_in, int epilogue, const float* bias, void* out, int64_t ldo, int split_out, int lo_off,
                void* stream);
/* X[M][N] (fp32, in place) += A . B^T + bias, then XN[M][ld_xn] (bf16) = LayerNorm(X) * gamma + beta with the engine's
 * eps: Block.forward's residual add (vit.py:110-111) fused with the LayerNorm that reads it next (:107 / :111).
 * bf16 engines only; N / 128 must be 1, 2, 3, 4 or 6 (one thread-block cluster spans a row). */
int vitocm_gemm_ln(vitocm_engine* e, const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K, const float* bias,
                   float* X, const float* gamma, const float* beta, void* XN, int64_t ld_xn, void* stream);
/* X[M][D] += gelu(XN . W1^T + bias1) . W2^T + bias2 in ONE kernel (Mlp.forward + the residual add, SSS/dino/vision_transformer.py:57-63,
 * :111): XN 16-bit [M][ld_xn], W1 [hidden][ldw1], W2 [D][ldw2] (K-major, the engine's 16-bit format), X fp32 [M][D].  The hidden
 * activations stay in shared / tensor memory.  D = 128 or 384, hidden a multiple of 128, engines with single 16-bit operands. */
int vitocm_mlp_fused(vitocm_engine* e, const void* XN, int64_t ld_xn, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2, int M,
                     int D, int hidden, const float* bias1, const float* bias2, float* X, void* stream);
/* Diagnostics: vitocm_mlp_fused that also records SM-clock stamps of the leader CTA of pair 0 on its second work item
 * (VITOCM_MLP_TL_ITEM): stamps int64 [64] (layout: MlpArgs::timeline in csrc/mlp_fused_sm100.cuh). */
int vitocm_mlp_fused_timeline(vitocm_engine* e, const void* XN, int64_t ld_xn, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2,
                              int M, int D, int hidden, const float* bias1, const float* bias2, float* X, int64_t* stamps, void* stream);
/* The second half of Block.forward in ONE kernel (SSS/dino/vision_transformer.py:88, :110-111, :57-63, and of the NEXT block :107 and
 * the qkv Linear of :80):  X += CTX . Wp^T + bias_p;  X += gelu(LayerNorm(X; ln2) . W1^T + bias1) . W2^T + bias2;  when next_ln_w is
 * not NULL, XN = LayerNorm(X; next_ln) in the engine's 16-bit format;  when Wqkv is not NULL as well, QKV = XN . Wqkv^T + bias_qkv is
 * written INSTEAD of XN (the normalised rows stay in shared memory).  CTX 16-bit [M][ld_ctx], Wp [D][ldwp], W1 [hidden][ldw1],
 * W2 [D][ldw2], Wqkv [3D][ldwqkv] (K-major), X fp32 [M][D] in place, XN 16-bit [M][ld_xn], QKV 16-bit [M][ld_qkv].  D = 128 or 384,
 * hidden a multiple of 128, engines with single 16-bit operands.  stamps: NULL, or int64 [64] SM-clock stamps (diagnostics; layout:
 * TailArgs::timeline in csrc/block_tail_sm100.cuh). */
int vitocm_block_tail(vitocm_engine* e, const void* CTX, int64_t ld_ctx, const void* Wp, int64_t ldwp, const float* bias_p, const float* ln2_w,
                      const float* ln2_b, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2, int M, int D, int hidden, const float* bias1,
                      const float* bias2, float* X, const float* next_ln_w, const float* next_ln_b, void* XN, int64_t ld_xn, const void* Wqkv,
                      int64_t ldwqkv, const float* bias_qkv, void* QKV, int64_t ld_qkv, int64_t* stamps, void* stream);
/* vitocm_block_tail in the form the forward runs after vitocm_finalize_weights: W1 / bias1 are taken to carry norm2's affine
 * parameters (W1 diag(ln2_w), bias1 + W1 ln2_b; ln2_w / ln2_b are not read) and, when Wqkv is not NULL, Wqkv / bias_qkv the next
 * norm1's (next_ln_w / next_ln_b are then only tested against NULL).  Without Wqkv, XN = LayerNorm(X; next_ln) keeps its affine
 * parameters.  Same arguments as vitocm_block_tail. */
int vitocm_block_tail_folded(vitocm_engine* e, const void* CTX, int64_t ld_ctx, const void* Wp, int64_t ldwp, const float* bias_p,
                             const float* ln2_w, const float* ln2_b, const void* W1, int64_t ldw1, const void* W2, int64_t ldw2, int M, int D,
                             int hidden, const float* bias1, const float* bias2, float* X, const float* next_ln_w, const float* next_ln_b,
                             void* XN, int64_t ld_xn, const void* Wqkv, int64_t ldwqkv, const float* bias_qkv, void* QKV, int64_t ld_qkv,
                             int64_t* stamps, void* stream);
/* ctx = MHSA(qkv) for B images of n_tokens tokens: qkv bf16 [B*N][ld] (columns [3][heads][head_dim]), ctx bf16 [B*N][ldo]. */
int vitocm_attention(vitocm_engine* e, const void* qkv, int64_t ld, int B, int n_tokens, void* ctx, int64_t ldo,
                     void* stream);
/* vitocm_attention for B images of n_tokens[i] (host int [B]) tokens packed back to back in qkv / ctx ([sum N_i] rows, no pad rows;
 * the kernels of vitocm_forward_cls_attn_varlen).  ws: device memory for the work-item table (16 bytes per item; a too small ws is
 * refused and the message names the size). */
int vitocm_attention_varlen(vitocm_engine* e, const void* qkv, int64_t ld, int B, const int* n_tokens, void* ctx, int64_t ldo, void* ws,
                            size_t ws_bytes, void* stream);
/* Diagnostics: vitocm_attention that also records SM-clock stamps of the CTAs of query tiles 0 and 1 of
 * (image 0, head 0): stamps int64 [2 cta][2 role: softmax warp 0, MMA thread][16 kv blocks][8 events]. */
int vitocm_attention_timeline(vitocm_engine* e, const void* qkv, int64_t ld, int B, int n_tokens, void* ctx, int64_t ldo,
                              int64_t* stamps, void* stream);
/* LayerNorm rows of X [M][D] fp32 with affine (gamma, beta) -> out bf16 [M][ldo] (hi | lo if split). */
int vitocm_layernorm(vitocm_engine* e, const float* X, const float* gamma, const float* beta, void* out_bf16,
                     int64_t ldo, int split, int lo_off, int M, void* stream);
/* ---- MIM training step (SSS/mim.py:153-182; model.py:71-77 under autograd).  16-bit engines: VITOCM_BF16 or VITOCM_FP16
 * (the fp32-parity mode is refused). ---- */

/* Master weights owned by the caller (training): `name` as in vitocm_load_weight, dev_data = DEVICE fp32, 16-byte aligned,
 * used in place (no copy) -- an optimizer updates it and vitocm_refresh_weights repacks the 16-bit operand copies (the engine's format) on
 * `stream` without synchronising.  The first use still needs one vitocm_finalize_weights. */
int vitocm_bind_weight(vitocm_engine* e, const char* name, float* dev_data, int64_t numel);
int vitocm_refresh_weights(vitocm_engine* e, void* stream);
/* Where vitocm_mim_backward and vitocm_encoder_backward ACCUMULATE dL/d(name) (fp32, same shape as the parameter; the caller zeroes it, like
 * optimizer.zero_grad(), mim.py:173).  NULL unbinds. */
int vitocm_bind_grad(vitocm_engine* e, const char* name, float* dev_grad);

/* Includes a slab of 8 depth B bytes (plus alignment) for the stochastic-depth scales of the _dp forwards. */
size_t vitocm_mim_train_workspace_bytes(const vitocm_engine* e, int B, int n_tokens);
/* MIM.forward (model.py:71-77) for one batch, keeping the activations the backward needs in ws (same arguments as
 * vitocm_mim_forward; the whole batch is one chunk).  = vitocm_mim_train_forward_dp with branch_scale NULL. */
int vitocm_mim_train_forward(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask,
                             float* x_rec, double* loss_sums, void* ws, size_t ws_bytes, void* stream);
/* The same with stochastic depth (DINO's DropPath, vit.py:101,110-111): branch_scale = DEVICE fp32 [depth][2][B], [l][0][b] the
 * scale of block l's attention branch for image b and [l][1][b] that of its MLP branch (0 or 1 / keep in training; any value is
 * applied): x += s (proj(...) + bias) and x += s (fc2(...) + bias).  The scales are copied into ws on the stream, and the backward on
 * this ws uses that copy: the gradient entering a branch is s dX, the residual path carries dX unscaled.  NULL = no drop path. */
int vitocm_mim_train_forward_dp(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, const float* mask,
                                float* x_rec, double* loss_sums, const float* branch_scale, void* ws, size_t ws_bytes, void* stream);
/* loss.backward() (mim.py:174) for the batch vitocm_mim_train_forward(_dp) just ran on the same ws (with its branch scales): gradients of
 * (*grad_scale) * loss (grad_scale = DEVICE pointer to the upstream gradient of the scalar loss, NULL = 1) are accumulated into the buffers bound with vitocm_bind_grad (all parameters except pos_embed);
 * dpos [N][D] fp32 is WRITTEN with the gradient of the (interpolated) position table passed to the forward.
 * Loss scale (fp16 engines): fp16's range would flush the loss gradient (~4e-7 at batch 32, 224^2) towards zero, so the backward
 * runs on gradients multiplied by S = 2^e, chosen on the device (no host sync) from the exponent of the loss gradient
 * *grad_scale / (3 (sum(mask) + 1e-5)) so that its magnitude times S lies in [1, 2); S = 1 if that is 0.  S and 1 / S are kept in
 * 8 bytes of ws.  Every parameter gradient and dpos are multiplied by 1 / S before they are written or accumulated, which is
 * exact: callers see the unscaled gradients, and a power-of-two grad_scale scales them exactly.  bf16 engines use no scale. */
int vitocm_mim_backward(vitocm_engine* e, const float* x, int B, int H, int W, const float* mask, const float* x_rec,
                        const double* loss_sums, const float* grad_scale, float* dpos, void* ws, size_t ws_bytes, void* stream);

/* Gradient buckets for an all-reduce that overlaps the backward (data-parallel training, SURVEY.md 8e): fills events[0..depth]
 * with cudaEvent_t handles owned by the engine; every later vitocm_mim_backward records events[l] on its stream once ALL
 * parameter gradients of transformer block l are complete (blocks finish last to first) and events[depth] once those of the
 * decoder and the final norm are.  The embedding gradients (cls / mask token, patch filter; pos via dpos) complete when the call's
 * last kernel does.  vitocm_stream_wait_event(stream, event) = cudaStreamWaitEvent, for callers without a CUDA binding. */
int vitocm_mim_backward_events(vitocm_engine* e, void** events, int n);
int vitocm_stream_wait_event(void* stream, void* event);

/* ---- Encoder training under any loss: fine-tuning (SSS/finetune.py, heads SSS/model.py:110-174) and DINO's linear evaluation on
 * get_intermediate_layers (vit.py:248-256).  16-bit engines only, no decoder weights needed; ws sized by
 * vitocm_mim_train_workspace_bytes(e, B, N). ---- */
/* forward_feats / get_intermediate_layers(x, n_out) (vit.py:198-223, 248-256) for one batch, keeping the activations the backward
 * needs in ws: feats [n_out][B][N][D] fp32 = norm(x_l) of the last n_out blocks (slab n_out - 1 = the last block), CLS row
 * included.  pos [N][D] fp32: the (interpolated) position table, as in vitocm_prepare_tokens. */
int vitocm_encoder_train_forward(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, int n_out, float* feats,
                                 void* ws, size_t ws_bytes, void* stream);
/* vitocm_encoder_train_forward with stochastic depth: branch_scale as in vitocm_mim_train_forward_dp (NULL = none). */
int vitocm_encoder_train_forward_dp(vitocm_engine* e, const float* x, int B, int H, int W, const float* pos, int n_out, float* feats,
                                    const float* branch_scale, void* ws, size_t ws_bytes, void* stream);
/* Backward of the vitocm_encoder_train_forward(_dp) that last ran on the same ws (with its branch scales), for the upstream gradient dfeats [n_out][B][N][D]
 * fp32 (DEVICE): parameter gradients are ACCUMULATED into the buffers bound with vitocm_bind_grad (every encoder parameter except
 * pos_embed; mask_token and the decoder are not touched), dpos [N][D] is WRITTEN, and so is dx [B][C][H][W] fp32 unless dx is NULL.
 * fp16 engines: S = 2^e is picked on the device from max |dfeats| so that max |dfeats| S lies in [1, 2) (S = 1 for an all-zero
 * upstream) and undone exactly as in vitocm_mim_backward.  The events of vitocm_mim_backward_events are recorded here too; with
 * n_out > 1 the gradients of norm.* complete with block depth - n_out + 1's event instead of events[depth].  The first call with
 * dx adds a transposed copy of the patch filter to the engine's repack (one extra refresh, then kept up to date by it). */
int vitocm_encoder_backward(vitocm_engine* e, const float* x, int B, int H, int W, int n_out, const float* dfeats, float* dpos,
                            float* dx, void* ws, size_t ws_bytes, void* stream);

/* torch.nn.utils.clip_grad_norm_ (mim.py:176), first half: out[0] = sum g^2 over a flat fp32 gradient buffer (fp64). */
int vitocm_grad_sumsq(const float* g, int64_t n, double* out, void* stream);
/* Second half, in place like the reference's call (mim.py:176): g <- g * min(1, max_norm / (sqrt(*sumsq) + 1e-6)), the coefficient
 * formed on the device from the sum of squares vitocm_grad_sumsq just wrote (no host sync). */
int vitocm_grad_clip(float* g, int64_t n, float max_norm, const double* sumsq, void* stream);
/* torch.optim.AdamW.step (the clip may also be folded in: max_norm > 0 with the sumsq of the CURRENT gradient)
 * Second half fused with torch.optim.AdamW.step (optimizer.py:73-75) over flat fp32 buffers of n elements:
 * g <- g * grad_scale * min(1, max_norm / (sqrt(*sumsq) * grad_scale + 1e-6)) (max_norm <= 0 or sumsq NULL: no clipping),
 * then the decoupled-weight-decay Adam update with bias correction for step number `step` (1-based); decay[i] != 0
 * selects weight decay per element (none for 1-D parameters and biases, optimizer.py:14-33). */
int vitocm_adamw_step(float* p, float* g, float* m, float* v, const uint8_t* decay, int64_t n, float lr, float beta1, float beta2,
                      float eps, float weight_decay, int step, float max_norm, float grad_scale, const double* sumsq, void* stream);

/* kernel-level: dW[R][C] (fp32) += G[M][R]^T . A[M][C], 16-bit row-major activations in the engine's format (bf16 or fp16; the weight
 * gradient of nn.Linear);
 * db[R] (fp32, or NULL) += column sums of G (its bias gradient, computed by the same tensor-core pass) */
int vitocm_wgrad(vitocm_engine* e, const void* G, int64_t ldg, const void* A, int64_t lda, int M, int R, int C, float* dW,
                 float* db, void* stream);
/* vitocm_attention that also returns lse2 [B][heads][Npad] = log2 sum_k exp(scale q.k); Npad = n_tokens rounded up to a
 * multiple of 128, pad rows hold +inf */
int vitocm_attention_fwd_lse(vitocm_engine* e, const void* qkv, int64_t ld, int B, int n_tokens, void* ctx, int64_t ldo,
                             float* lse2, void* stream);
/* backward of vitocm_attention on bf16 or fp16 engines (operands and dqkv in the engine's format): dqkv [B*N][ldq] (columns
 * [3][heads][head_dim]) from dctx; scratch: delta [B][heads][Npad] fp32,
 * dqacc [B*N][D] fp32 (zero on entry, zero again on return) */
int vitocm_attention_bwd(vitocm_engine* e, const void* qkv, int64_t ld, const void* ctx, const void* dctx, int64_t ldc,
                         const float* lse2, float* delta, float* dqacc, void* dqkv, int64_t ldq, int B, int n_tokens,
                         void* stream);
/* kernel-level: out[M][N] = (dY[M][K] . Wt[N][K]^T) * gelu'(pre[M][N]), all 16-bit in the engine's format (bf16 or fp16 engines):
 * the input gradient of fc2 through the GELU as the training step computes it, the derivative of the GELU form the engine's
 * forward uses.  pre [M][ld_pre] 16-byte aligned, ld_pre a multiple of 8 (the step passes HP + hidden with ld_pre = 2 hidden). */
int vitocm_gemm_dgelu(vitocm_engine* e, const void* dY, int64_t ldy, const void* Wt, int64_t ldw, int M, int N, int K, const void* pre,
                      int64_t ld_pre, void* out, int64_t ldo, void* stream);
/* kernel-level: nn.LayerNorm backward with the engine's eps for rows X [M][D] fp32 and dy [M][ld_dy] (16-bit, the engine's format):
 * dX [M][D] fp32 = (accumulate ? dX : 0) + dx;  dXb [M][D] = 16-bit(dX);  dgamma[D] += sum dy xhat;  dbeta[D] += sum dy;
 * dbias_out[D] (or NULL) += column sums of the new dX.  fp16 engines: lscale = DEVICE [S, 1 / S], dy and dX carry S and the three
 * column sums are multiplied by 1 / S (NULL: 1); bf16 engines ignore it.  D % 4 == 0, D <= 1024. */
int vitocm_layernorm_bwd(vitocm_engine* e, const float* X, const void* dy, int64_t ld_dy, const float* gamma, float* dX, void* dXb,
                         float* dgamma, float* dbeta, float* dbias_out, int accumulate, int M, int D, const float* lscale, void* stream);
/* kernel-level: vitocm_layernorm_bwd where dXb and the dbias_out column sums use s dX with s = row_scale[row / rows_per_scale] (DEVICE
 * fp32; the stochastic-depth scale of the branch this gradient enters); dX, dgamma and dbeta are those of vitocm_layernorm_bwd.
 * row_scale NULL = vitocm_layernorm_bwd. */
int vitocm_layernorm_bwd_scaled(vitocm_engine* e, const float* X, const void* dy, int64_t ld_dy, const float* gamma, float* dX, void* dXb,
                                float* dgamma, float* dbeta, float* dbias_out, int accumulate, int M, int D, const float* lscale,
                                const float* row_scale, int rows_per_scale, void* stream);
/* kernel-level: vitocm_gemm with epilogue 2, X[M][ldx] (fp32, in place) += (A . B^T + bias) * row_scale[row / rows_per_scale]
 * (DEVICE fp32; the proj / fc2 residual add under stochastic depth).  row_scale NULL = vitocm_gemm with epilogue 2. */
int vitocm_gemm_resid_scaled(vitocm_engine* e, const void* A, int64_t lda, const void* B, int64_t ldb, int M, int N, int K, const float* bias,
                             float* X, int64_t ldx, const float* row_scale, int rows_per_scale, void* stream);
/* kernel-level: the loss gradient of vitocm_mim_backward, dY [B (n + 1)][C p^2] (16-bit, the engine's format; C and p from the engine,
 * n = (H / p) (W / p)) = *grad_scale * mask * sign(x_rec - x) / ((loss_sums[1] + 1e-5) C) through PixelShuffle, 0 at ties and in CLS
 * rows.  fp16 engines multiply it by the loss scale S described at vitocm_mim_backward and write [S, 1 / S] to lscale (DEVICE, or
 * NULL).  16-bit engines only. */
int vitocm_mim_loss_bwd(vitocm_engine* e, const float* x, const float* x_rec, const float* mask, const double* loss_sums,
                        const float* grad_scale, int B, int H, int W, void* dY, float* lscale, void* stream);

/* Diagnostics: SM-clock stamps of one CTA of the last vitocm_attention_bwd run under VITOCM_ABW_DEBUG=2: host int64
 * [role: softmax warp 0, MMA thread][query tile < 8][event < 8]. */
int vitocm_debug_abw_timeline(int64_t* host_out);

/* Optional per-kernel-class device timing: when enabled every launch is bracketed by CUDA events on
 * its own stream; vitocm_profile_read synchronises, sums milliseconds and launch counts per class
 * (vitocm_profile_classes() slots, names from vitocm_profile_class_name) and clears the log. */
int vitocm_profile_enable(int on);
int vitocm_profile_classes(void);
const char* vitocm_profile_class_name(int cls);
int vitocm_profile_read(double* ms, int64_t* counts, int nclasses);
/* number of kernels launched by this library on the calling process since load (gpu_launches) */
int64_t vitocm_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VITOCM_H_ */
