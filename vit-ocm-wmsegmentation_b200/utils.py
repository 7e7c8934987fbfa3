"""Drop-in for the hot-path half of the reference's ``utils.py`` (eval / PGT flavour):
``compute_attention`` (SSS/utils.py:229-235), ``min_max_normalize`` (:55-60), ``threshold``
(:62-115), the plain-tiling ``concat_crops`` (:304-317), ``concat_crops_overlap`` (:319-347) and
``sliding_window`` (:349-362), plus ``attention_masks`` / ``cropped_attention_masks`` -- the batched,
device-resident versions of the per-image loop body at SSS/eval.py:136-173 (`--crop 1` and `--crop 4|16`).

All arithmetic runs in libvitocm.so kernels; torch is used for device buffers only.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import _lib
from ._lib import check, cur_stream, ptr


def _dev():
    if not torch.cuda.is_available():
        raise _lib.VitocmError("vitocm needs a CUDA device (B200, sm_100a); there is no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def head_mean_maps(cls_rows: torch.Tensor, per_tile_minmax255: bool = False) -> torch.Tensor:
    """[T, heads, N] CLS rows -> [T, N-1] low-res maps (head mean; optionally the per-tile
    min-max * 255 of SSS/sw_processing.py:253-254)."""
    cls_rows = cls_rows.contiguous()
    T, H, N = cls_rows.shape
    out = torch.empty(T, N - 1, dtype=torch.float32, device=cls_rows.device)
    check(_lib.load_library().vitocm_head_mean(ptr(cls_rows), ptr(out), T, H, N, int(per_tile_minmax255), cur_stream()))
    return out


def cummass_threshold(cls_rows: torch.Tensor, threshold: float, w_featmap: int | None = None, h_featmap: int | None = None,
                      patch_size: int | None = None):
    """The `--threshold` mode (flag at SSS/eval.py:33-34; semantics of upstream DINO's visualize_attention.py: "we keep only a
    certain percentage of the mass"): per tile and head, the patches are sorted by CLS attention, normalised to unit mass, and
    those whose ascending cumulative mass exceeds 1 - threshold are kept.  cls_rows [T, heads, N] (e.g. model.cls_attention_rows(x))
    -> mask [T, heads, N - 1] uint8 in {0, 1}; with (w_featmap, h_featmap, patch_size) also the nearest-upsampled float masks
    [T, heads, w*p, h*p] that visualize_attention.py displays.  Everything on the device (one block per (tile, head): bitonic
    sort + shuffle scan).  Not under /root/reference: parity unpinned by the reference (oracle/post_oracle.py cummass_threshold)."""
    cls_rows = cls_rows.contiguous()
    T, H, N = cls_rows.shape
    mask = torch.empty(T, H, N - 1, dtype=torch.uint8, device=cls_rows.device)
    up = None
    lh = lw = p = 0
    if patch_size is not None:
        lh, lw, p = int(w_featmap), int(h_featmap), int(patch_size)
        up = torch.empty(T, H, lh * p, lw * p, dtype=torch.float32, device=cls_rows.device)
    check(_lib.load_library().vitocm_attn_cummass(ptr(cls_rows), T, H, N, float(threshold), ptr(mask), ptr(up), lh, lw, p, cur_stream()))
    return (mask, up) if up is not None else mask


def compute_attention(attentions, query, w_featmap, h_featmap, patch_size):
    """SSS/utils.py:229-235: attention of `query` for batch element 0, per head, nearest-upsampled
    by the patch size, as a host numpy array [nh, w*p, h*p]; returns (array, nh)."""
    a0 = attentions[0]
    nh = a0.shape[1]
    row = a0[0, :, query, 1:]                       # LazyAttention serves query == 0 from the CLS rows
    row = row.reshape(nh, w_featmap, h_featmap)
    up = row.repeat_interleave(patch_size, dim=1).repeat_interleave(patch_size, dim=2)   # nearest: a copy, no arithmetic
    return up.cpu().numpy(), nh


def min_max_normalize(image):
    """SSS/utils.py:55-60 (host helper kept for callers; `threshold` does this on the device)."""
    mn, mx = np.min(image), np.max(image)
    if mx == mn:
        return image
    return (image - mn) / (mx - mn)


def _save_gray(path, arr):
    from PIL import Image
    Image.fromarray(np.asarray(arr, dtype=np.uint8)).save(path)


def _save_threshold_images(output_directory, name, th, th2, th3, result, att_u8):
    """The five files of SSS/utils.py:102-114 (= SSS/sw_processing.py:68-80), same names and places.  `temp.png` is the
    normalised attention as a gray image (the reference sends the float map through matplotlib's default colour map)."""
    sub = (name + "/") if name is not None else ""
    os.makedirs(os.path.join(output_directory, sub) or ".", exist_ok=True)
    _save_gray(os.path.join(output_directory, sub, "OTSU_th_average.png"), th)
    _save_gray(os.path.join(output_directory, "OTSU_th_original.png"), th2)
    _save_gray(os.path.join(output_directory, "weighted_iamge_attention.png"), result)
    _save_gray(os.path.join(output_directory, "heatmap_otsu_attention.png"), th3)
    _save_gray(os.path.join(output_directory, "temp.png"), att_u8)


def threshold(img, attention, output_directory="", save=True, name=None):
    """SSS/utils.py:62-115.  img: PIL "L" image or uint8 array [S, S]; attention: float array [S, S].
    Returns (th, th2, th3) uint8 {0,255} host arrays: Otsu of the 0.6/0.4 image/attention blend
    ("ours"), Otsu of the image, Otsu of the attention heat-map ("heatmap_threshold")."""
    dev = _dev()
    img_np = np.ascontiguousarray(np.array(img), dtype=np.uint8)
    att_np = np.ascontiguousarray(np.asarray(attention), dtype=np.float32)
    if img_np.ndim != 2 or img_np.shape != att_np.shape or img_np.shape[0] != img_np.shape[1]:
        raise ValueError("threshold expects a square gray image and an attention map of the same size")
    S = img_np.shape[0]
    d_img = torch.from_numpy(img_np).to(dev)
    d_att = torch.from_numpy(att_np).to(dev)
    masks = torch.empty(1, 3, S, S, dtype=torch.uint8, device=dev)
    thr = torch.empty(1, 3, dtype=torch.int32, device=dev)
    aux = torch.empty(1, 2, S, S, dtype=torch.uint8, device=dev) if save else None
    check(_lib.load_library().vitocm_tile_threshold_aux(None, None, 1, 1, S, 1, 1, ptr(masks), ptr(thr), None, ptr(d_att),
                                                        ptr(d_img), ptr(aux), cur_stream()))
    th, th2, th3 = (m.cpu().numpy() for m in masks[0])
    if save:
        _save_threshold_images(output_directory, name, th, th2, th3, aux[0, 0].cpu().numpy(), aux[0, 1].cpu().numpy())
    return th, th2, th3


def concat_crops(crops):
    """SSS/utils.py:304-317: non-overlapping row-major tiling of n*n crops (pure data movement)."""
    n = int(np.sqrt(len(crops)))
    rows = [np.concatenate(list(crops[i * n:(i + 1) * n]), axis=1) for i in range(n)]
    return np.concatenate(rows, axis=0)


@torch.no_grad()
def attention_masks(model, x: torch.Tensor, return_attention: bool = False):
    """Device-resident, batched SSS/eval.py:136-173 (`--crop 1`): for every image of x [B, C, S, S]
    the last-layer CLS attention -> head mean -> bilinear x p -> utils.threshold.
    Returns dict(masks [B, 3, S, S] u8 (ours, otsu, heatmap), thresholds [B, 3] int32, lowres [B, h, w]
    [, attention [B, S, S]])."""
    rows = model.cls_attention_rows(x)
    B, _, S, S2 = x.shape
    if S != S2:
        raise ValueError("attention_masks expects square tiles")
    p = model.patch_embed.patch_size
    low = head_mean_maps(rows, per_tile_minmax255=False)
    lh = lw = S // p
    masks = torch.empty(B, 3, S, S, dtype=torch.uint8, device=x.device)
    thr = torch.empty(B, 3, dtype=torch.int32, device=x.device)
    att = torch.empty(B, S, S, dtype=torch.float32, device=x.device) if return_attention else None
    xx = x.detach().to(torch.float32).contiguous()
    check(_lib.load_library().vitocm_tile_threshold(ptr(low), ptr(xx), B, x.shape[1], S, lh, lw, ptr(masks), ptr(thr),
                                                    ptr(att), None, None, cur_stream()))
    out = dict(masks=masks, thresholds=thr, lowres=low.view(B, lh, lw), cls_rows=rows)
    if return_attention:
        out["attention"] = att
    return out


@torch.no_grad()
def attention_masks_varlen(model, images, return_attention: bool = False):
    """attention_masks for a list of square images of different sizes (the `--crop 1` eval body per image, SSS/eval.py:136-173, whose
    resize is square, :171), in one forward (VisionTransformer.cls_attention_rows_varlen) and one launch per post-processing step.
    images: CUDA tensors [C, S_i, S_i].  Returns dict(masks = list of [3, S_i, S_i] u8, thresholds [B, 3] int32, lowres = list of
    [h_i, w_i], cls_rows = list of [heads, N_i] [, attention = list of [S_i, S_i]]), each entry equal to attention_masks(x_i[None])'s."""
    for i, im in enumerate(images):
        if im.dim() != 3 or im.shape[1] != im.shape[2]:
            raise ValueError(f"attention_masks_varlen expects square [C, S, S] images (image {i} is {tuple(im.shape)})")
    packed, plan = model._cls_rows_varlen_packed(images)
    heads = model.num_heads
    rows = [packed[heads * t0:heads * (t0 + n)].view(heads, n) for t0, n in zip(plan["row0"], plan["n"])]
    p = model.patch_embed.patch_size
    B, dev = len(images), images[0].device
    sides = [int(im.shape[1]) for im in images]
    npatch = [(s // p) ** 2 for s in sides]
    poff = torch.tensor([0] + npatch, dtype=torch.int64).cumsum(0)
    pix = torch.tensor([0] + [s * s for s in sides], dtype=torch.int64).cumsum(0)
    low = torch.empty(int(poff[-1]), dtype=torch.float32, device=dev)
    lib = _lib.load_library()
    poff_d = poff.to(torch.int32).to(dev)
    check(lib.vitocm_head_mean_varlen(ptr(packed), ptr(low), B, heads, ptr(poff_d), 0, cur_stream()))
    geo = torch.tensor([[s, s // p, int(poff[i]), int(pix[i])] for i, s in enumerate(sides)], dtype=torch.int32).to(dev)
    masks = torch.empty(3 * int(pix[-1]), dtype=torch.uint8, device=dev)
    thr = torch.empty(B, 3, dtype=torch.int32, device=dev)
    att = torch.empty(int(pix[-1]), dtype=torch.float32, device=dev) if return_attention else None
    C = images[0].shape[0]
    xx = torch.cat([im.detach().to(torch.float32).reshape(-1) for im in images])
    check(lib.vitocm_tile_threshold_varlen(ptr(low), ptr(xx), B, C, ptr(geo), ptr(masks), ptr(thr), ptr(att), cur_stream()))
    out = dict(masks=[masks[3 * int(pix[i]):3 * int(pix[i + 1])].view(3, s, s) for i, s in enumerate(sides)], thresholds=thr,
               lowres=[low[int(poff[i]):int(poff[i + 1])].view(s // p, s // p) for i, s in enumerate(sides)], cls_rows=rows)
    if return_attention:
        out["attention"] = [att[int(pix[i]):int(pix[i + 1])].view(s, s) for i, s in enumerate(sides)]
    return out


def concat_crops_overlap(crops, stride):
    """SSS/utils.py:319-347: n x n crops overlapping by 2*stride; overlaps are `a // 2 + b // 2` (floor halves), along x
    inside each strip and then along y, the last strip being appended unblended.  float crops accumulate in float32,
    uint8 crops in uint8, as the reference's dtypes do.  Host arrays in and out; the fold runs on the device."""
    dev = _dev()
    n = int(np.sqrt(len(crops)))
    first = np.asarray(crops[0])
    W = first.shape[0]
    lib = _lib.load_library()
    E = W + (n - 1) * (W - 2 * int(stride))
    if first.dtype == np.uint8:
        stack = np.ascontiguousarray(np.stack([np.asarray(c) for c in crops[:n * n]]), dtype=np.uint8)
        squeeze = stack.ndim == 3
        if squeeze:
            stack = stack[..., None]
        C = stack.shape[-1]
        d = torch.from_numpy(stack).to(dev)
        out = torch.empty(max(E, 0), max(E, 0), C, dtype=torch.uint8, device=dev)
        check(lib.vitocm_concat_crops_overlap_u8(ptr(d), n, W, int(stride), C, ptr(out), cur_stream()))
        res = out.cpu().numpy()
        return res[..., 0] if squeeze else res
    stack = np.ascontiguousarray(np.stack([np.asarray(c, dtype=np.float32) for c in crops[:n * n]]))
    d = torch.from_numpy(stack).to(dev)
    out = torch.empty(max(E, 0), max(E, 0), dtype=torch.float32, device=dev)
    check(lib.vitocm_concat_crops_overlap_f32(ptr(d), n, W, int(stride), ptr(out), cur_stream()))
    return out.cpu().numpy()


def sliding_window(image, window_size, stride):
    """SSS/utils.py:349-362 (note the argument order: the mosaic script's twin takes (image, stride, window_size)).
    image: PIL image or uint8 array [H, W(, C)] -> list of uint8 crops, row-major, zero padded beyond the image."""
    dev = _dev()
    arr = np.ascontiguousarray(np.array(image), dtype=np.uint8)
    squeeze = arr.ndim == 2
    if squeeze:
        arr = arr[:, :, None]
    H, W, C = arr.shape
    # `height, width = image.size` unpacks PIL's (width, height): y runs over the width (:351)
    ny, nx = len(range(0, W - stride * 2, stride)), len(range(0, H - stride * 2, stride))
    if ny <= 0 or nx <= 0:
        return []
    d_img = torch.from_numpy(arr).to(dev)
    crops = torch.empty(ny * nx, window_size, window_size, C, dtype=torch.uint8, device=dev)
    check(_lib.load_library().vitocm_crop_u8(ptr(d_img), H, W, C, ny, nx, window_size, stride, ptr(crops), cur_stream()))
    out = crops.cpu().numpy()
    if squeeze:
        out = out[..., 0]
    return [out[i] for i in range(out.shape[0])]


@torch.no_grad()
def cropped_attention_masks(model, images: torch.Tensor, return_attention: bool = False):
    """Device-resident, batched SSS/eval.py:145-173 (`--crop 4|16`, data.py:85-125): every image arrives as cr*cr
    equal crops, images [B, cr*cr, C, s, s]; each crop goes through the ViT on its own, the head-mean CLS maps and
    channel 0 of the crops are tiled back (plain `concat_crops`, :160-161), the tiled map is upsampled bilinearly
    over the whole image (:169-171) and thresholded against the tiled image (`utils.threshold`).
    Returns dict(masks [B, 3, S, S] u8 (ours, otsu, heatmap), thresholds [B, 3], lowres [B, cr*h, cr*w], image
    [B, 1, S, S] [, attention [B, S, S]]) with S = cr * s."""
    if images.dim() != 5 or images.shape[-1] != images.shape[-2]:
        raise ValueError("cropped_attention_masks expects [B, crops, C, s, s]")
    B, ncrop, C, s, _ = images.shape
    cr = int(np.sqrt(ncrop))
    if cr * cr != ncrop:
        raise ValueError("the number of crops must be a square (4, 16, ...)")
    lib = _lib.load_library()
    p = model.patch_embed.patch_size
    xx = images.detach().to(torch.float32).contiguous()
    rows = model.cls_attention_rows(xx.view(B * ncrop, C, s, s))
    low = head_mean_maps(rows, per_tile_minmax255=False)                      # [B*ncrop, h*h]
    h = s // p
    S = cr * s
    low_t = torch.empty(B, cr * h, cr * h, dtype=torch.float32, device=xx.device)
    check(lib.vitocm_concat_grid_f32(ptr(low), B, cr, 1, 0, h, h, ptr(low_t), cur_stream()))
    img_t = torch.empty(B, 1, S, S, dtype=torch.float32, device=xx.device)
    check(lib.vitocm_concat_grid_f32(ptr(xx), B, cr, C, 0, s, s, ptr(img_t), cur_stream()))
    masks = torch.empty(B, 3, S, S, dtype=torch.uint8, device=xx.device)
    thr = torch.empty(B, 3, dtype=torch.int32, device=xx.device)
    att = torch.empty(B, S, S, dtype=torch.float32, device=xx.device) if return_attention else None
    check(lib.vitocm_tile_threshold(ptr(low_t), ptr(img_t), B, 1, S, cr * h, cr * h, ptr(masks), ptr(thr), ptr(att), None, None,
                                    cur_stream()))
    out = dict(masks=masks, thresholds=thr, lowres=low_t, image=img_t, cls_rows=rows)
    if return_attention:
        out["attention"] = att
    return out


# ----------------------------------------------------------------------------- checkpoints (SURVEY.md 8f rank 4)
def get_grad_norm(parameters, norm_type=2):
    """SSS/utils.py:363-373: total gradient norm over `parameters` (a tensor, an iterable of parameters, or a
    FusedAdamW / MIM whose gradients live in one flat buffer -- then a single reduction kernel)."""
    flat = getattr(getattr(parameters, "mim", parameters), "_gflat", None)
    lib = _lib.load_library()
    acc = None
    if flat is not None and float(norm_type) == 2.0:
        grads = [flat]
    else:
        if isinstance(parameters, torch.Tensor):
            parameters = [parameters]
        grads = [p.grad.detach() for p in parameters if p.grad is not None]
    if float(norm_type) != 2.0:
        raise NotImplementedError("vitocm get_grad_norm: only the 2-norm (the reference's call, SSS/mim.py:178,186) is on the device")
    total = 0.0
    for g in grads:
        g = g.to(torch.float32).contiguous()
        if g.data_ptr() % 16:
            g = g.clone()
        acc = torch.empty(1, dtype=torch.float64, device=g.device)
        check(lib.vitocm_grad_sumsq(ptr(g), g.numel(), ptr(acc), cur_stream()))
        total += float(acc.item())
    return total ** 0.5


def save_checkpoint(config, epoch, model, max_accuracy, optimizer, lr_scheduler, logger):
    """SSS/utils.py:375-385: {'model', 'optimizer', 'lr_scheduler', 'max_accuracy', 'epoch', 'config'} ->
    config.OUTPUT/ckpt_epoch_{epoch}.pth.  The reference passes the ENCODER (SSS/mim.py:123), so 'model' carries the
    plain ViT keys that eval.py / sw_processing.py load; tensors are stored as ordinary fp32 CPU tensors (the flat
    training buffers and the engine's repacked bf16 copies never reach the file)."""
    save_state = {'model': {k: v.detach().to("cpu", copy=True) for k, v in model.state_dict().items()},
                  'optimizer': optimizer.state_dict(),
                  'lr_scheduler': lr_scheduler.state_dict(),
                  'max_accuracy': max_accuracy,
                  'epoch': epoch,
                  'config': config}
    save_path = os.path.join(config.OUTPUT, f'ckpt_epoch_{epoch}.pth')
    if logger is not None:
        logger.info(f"{save_path} saving......")
    torch.save(save_state, save_path)
    if logger is not None:
        logger.info(f"{save_path} saved !!!")
    return save_path


def load_pretrained_weights(model, pretrained_weights, checkpoint_key=None):
    """The checkpoint branch of SSS/eval.py:67-77 (= sw_processing.py:187-197, analyse_attention.py:61-71): torch.load
    on the CPU, optional `checkpoint_key`, the `module.` / `backbone.` prefix strips, then
    ``model.load_state_dict(state_dict["model"], strict=False)``.  Returns the load message.  The engine picks the new
    values up by itself (parameter versions change -> weights are repacked before the next forward)."""
    state_dict = torch.load(pretrained_weights, map_location="cpu", weights_only=False)
    if checkpoint_key is not None and checkpoint_key in state_dict:
        state_dict = state_dict[checkpoint_key]
    state_dict = {k.replace("module.", ""): v for k, v in state_dict.items()}
    state_dict = {k.replace("backbone.", ""): v for k, v in state_dict.items()}
    return model.load_state_dict(state_dict["model"], strict=False)
