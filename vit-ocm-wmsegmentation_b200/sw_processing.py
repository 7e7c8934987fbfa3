"""Drop-in for the reference's mosaic script ``sw_processing.py`` on B200.

Function-level mirrors (same names / arguments as the reference, host arrays in and out):
  ``sliding_window`` (SSS/sw_processing.py:151-163), ``concat_crops`` + blends (:113-149),
  ``threshold`` (:37-81).
Device pipeline: ``MosaicSegmenter`` = the ``__main__`` body (:223-262) -- sliding window, per-crop
ViT CLS attention, head mean, per-tile min-max, resize pair, ramp-blended stitching, global
min-max, img*att, Otsu -- with the mosaic, every tile and the masks resident in HBM, tiles
batched through the engine, and (optionally) sharded over ranks of a torch.distributed group:
each rank runs the ViT on a contiguous slice of the tiles, the low-res maps are all-gathered,
each rank thresholds a band of output rows, {min, max, histograms} are all-reduced, and the mask
bands are gathered on rank 0 ("only a final mask gather").
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from ._lib import check, cur_stream, ptr
from .utils import _dev, _save_threshold_images, head_mean_maps


def _wtab(window_size: int, stride: int, device) -> torch.Tensor:
    """numpy.linspace(1, 0, window - stride) -- the blend ramp of :138/:145, bit-identical."""
    return torch.from_numpy(np.linspace(1, 0, window_size - stride)).to(device)


def grid_size(size: int, stride: int) -> int:
    """Number of window origins per axis: len(range(0, size - 2*stride, stride)) (:156-157)."""
    return len(range(0, size - stride * 2, stride))


def mosaic_grid(height: int, width: int, stride: int, window: int):
    """Window grid and stitched extent of a [height, width] mosaic: ((ny, nx), (Ey, Ex)).  Rows of windows come from the height,
    columns from the width; window t (row-major) has origin ((t // nx) * stride, (t % nx) * stride)."""
    ny, nx = grid_size(height, stride), grid_size(width, stride)
    return (ny, nx), ((ny - 1) * stride + window, (nx - 1) * stride + window)


# ----------------------------------------------------------------------------- function mirrors
def sliding_window(image, stride=128, window_size=384):
    """SSS/sw_processing.py:151-163.  image: PIL image or uint8 array [H, W(, C)].
    Returns the list of uint8 crops (row-major; zero padded beyond the image like PIL's crop)."""
    dev = _dev()
    arr = np.ascontiguousarray(np.array(image), dtype=np.uint8)
    squeeze = arr.ndim == 2
    if squeeze:
        arr = arr[:, :, None]
    H, W, C = arr.shape
    # the reference unpacks PIL's (width, height) as `height, width`: y iterates over the width
    ny, nx = grid_size(W, stride), grid_size(H, stride)
    if ny <= 0 or nx <= 0:
        return []
    d_img = torch.from_numpy(arr).to(dev)
    crops = torch.empty(ny * nx, window_size, window_size, C, dtype=torch.uint8, device=dev)
    check(_lib.load_library().vitocm_crop_u8(ptr(d_img), H, W, C, ny, nx, window_size, stride, ptr(crops), cur_stream()))
    out = crops.cpu().numpy()
    if squeeze:
        out = out[..., 0]
    return [out[i] for i in range(out.shape[0])]


def concat_crops(crops, stride, window_size, grid=None):
    """SSS/sw_processing.py:113-134: row-major n x n grid of crops, overlapping by window - stride,
    seams blended with a linear ramp, first along x inside each strip then along y.  float32 crops
    accumulate in float32, uint8 crops truncate at every seam -- as the reference's dtypes do.
    grid: (ny, nx) stitches ny strips of nx crops into [(ny-1) S + W, (nx-1) S + W] (a rectangular mosaic, which the
    reference cannot stitch: it takes n = sqrt(len(crops))); None infers the square grid as the reference does."""
    dev = _dev()
    if grid is None:
        n = int(np.sqrt(len(crops)))
        ny = nx = n
    else:
        ny, nx = int(grid[0]), int(grid[1])
        if ny < 1 or nx < 1 or len(crops) < ny * nx:
            raise ValueError(f"concat_crops: a {ny} x {nx} grid needs {max(ny, 0) * max(nx, 0)} crops, got {len(crops)}")
    first = np.asarray(crops[0])
    lib = _lib.load_library()
    wtab = _wtab(window_size, stride, dev)
    Ey, Ex = (ny - 1) * stride + window_size, (nx - 1) * stride + window_size
    if first.dtype == np.uint8:
        stack = np.ascontiguousarray(np.stack([np.asarray(c) for c in crops[:ny * nx]]), dtype=np.uint8)
        squeeze = stack.ndim == 3
        if squeeze:
            stack = stack[..., None]
        C = stack.shape[-1]
        d = torch.from_numpy(stack).to(dev)
        out = torch.empty(Ey, Ex, C, dtype=torch.uint8, device=dev)
        check(lib.vitocm_concat_crops_grid_u8(ptr(d), ny, nx, window_size, stride, C, ptr(wtab), ptr(out), cur_stream()))
        res = out.cpu().numpy()
        return res[..., 0] if squeeze else res
    stack = np.ascontiguousarray(np.stack([np.asarray(c, dtype=np.float32) for c in crops[:ny * nx]]))
    d = torch.from_numpy(stack).to(dev)
    out = torch.empty(Ey, Ex, dtype=torch.float32, device=dev)
    check(lib.vitocm_concat_crops_grid_f32(ptr(d), ny, nx, window_size, stride, ptr(wtab), ptr(out), cur_stream()))
    return out.cpu().numpy()


def _threshold_device(lib, lowres, geom, wtab, gray, map_in, y0, y1, group=None, want=("th", "th3"), gray_base=None):
    """Three passes over output rows [y0, y1): stitched map + min/max -> histograms -> Otsu -> masks.  The stitched map is
    evaluated once (pass 1 keeps it as an fp32 band, passes 2 and 3 read it back).  geom = (ny, nx, W, S, lh, lw).  gray: full
    [Ey, Ex] uint8 tensor, or None with gray_base = address such that row Y of the stitched image starts at gray_base + Y * Ex
    (a band buffer shifted by y0 rows)."""
    ny, nx, W, S, lh, lw = geom
    E = (nx - 1) * S + W            # row length Ex
    dev = lowres.device if lowres is not None else map_in.device
    st = cur_stream()
    gray_p = ptr(gray) if gray is not None else gray_base
    rows = y1 - y0
    minmax = torch.empty(2, dtype=torch.int32, device=dev)
    check(lib.vitocm_minmax_init(ptr(minmax), st))
    band_map = None
    if map_in is None:
        # absolute-row addressing into a band-sized buffer: base = data_ptr - y0 * E * 4 (never dereferenced outside [y0, y1))
        band_map = torch.empty(max(rows, 1), E, dtype=torch.float32, device=dev)
        map_p = band_map.data_ptr() - y0 * E * 4
        check(lib.vitocm_stitch_minmax_grid(ptr(lowres), ny, nx, W, S, lh, lw, ptr(wtab), y0, y1, ptr(minmax), map_p, None, st))
    else:
        map_p = ptr(map_in)
        check(lib.vitocm_stitch_minmax_grid(None, ny, nx, W, S, lh, lw, ptr(wtab), y0, y1, ptr(minmax), None, map_p, st))
    if group is not None:
        allreduce_minmax(minmax, group)
    hists = torch.zeros(3, 256, dtype=torch.int64, device=dev)
    check(lib.vitocm_stitch_hist_grid(ptr(lowres), ny, nx, W, S, lh, lw, ptr(wtab), gray_p, ptr(minmax), y0, y1, ptr(hists), map_p, st))
    if group is not None:
        import torch.distributed as dist
        dist.all_reduce(hists, op=dist.ReduceOp.SUM, group=group)
    thr = torch.empty(3, dtype=torch.int32, device=dev)
    check(lib.vitocm_otsu(ptr(hists), 3, ptr(thr), st))
    masks = {k: torch.empty(rows, E, dtype=torch.uint8, device=dev) for k in want}
    check(lib.vitocm_stitch_mask_grid(ptr(lowres), ny, nx, W, S, lh, lw, ptr(wtab), gray_p, ptr(minmax), ptr(thr), y0, y1,
                                      ptr(masks.get("th")), ptr(masks.get("th2")), ptr(masks.get("th3")), map_p, st))
    return masks, thr, minmax, hists


def threshold(img, attention, output_directory="", save=True, name=None):
    """SSS/sw_processing.py:37-81.  img: PIL "L" image or uint8 array [H, W]; attention: float array
    [H, W] (the stitched map).  Returns (th, th2, th3): Otsu of img * normalised attention, Otsu of
    the image (the reference uses skimage's Otsu for this off-path output; OpenCV's rule here), Otsu
    of the attention heat-map."""
    dev = _dev()
    img_np = np.ascontiguousarray(np.array(img), dtype=np.uint8)
    att_np = np.ascontiguousarray(np.asarray(attention), dtype=np.float32)
    if img_np.shape != att_np.shape or img_np.ndim != 2:
        raise ValueError("threshold expects a gray image and an attention map of the same 2-D shape")
    H, W = img_np.shape
    gray = torch.from_numpy(img_np).to(dev)
    amap = torch.from_numpy(att_np).to(dev)
    # the passes read the caller's map (map_in): the geometry only has to give the extent H x W.  A square uses a single "tile"
    # covering it (W = E; S only has to be < W); a rectangle a grid of 2-pixel windows at stride 1 (extent (ny-1) + 2 per axis)
    geom = (1, 1, H, H - 1 if H > 1 else 1, 1, 1) if H == W else (H - 1, W - 1, 2, 1, 1, 1)
    wtab = torch.zeros(max(geom[2] - geom[3], 1), dtype=torch.float64, device=dev)
    lib = _lib.load_library()
    masks, thr, minmax, _ = _threshold_device(lib, None, geom, wtab, gray, amap, 0, H, want=("th", "th2", "th3"))
    th, th2, th3 = (masks[k].cpu().numpy() for k in ("th", "th2", "th3"))
    if save:
        result = torch.empty(H, W, dtype=torch.uint8, device=dev)
        att_u8 = torch.empty(H, W, dtype=torch.uint8, device=dev)
        check(lib.vitocm_stitch_result_grid(None, *geom, ptr(wtab), ptr(gray), ptr(minmax), 0, H,
                                            ptr(result), ptr(att_u8), ptr(amap), cur_stream()))
        _save_threshold_images(output_directory, name, th, th2, th3, result.cpu().numpy(), att_u8.cpu().numpy())
    return th, th2, th3


# ----------------------------------------------------------------------------- device pipeline
def shard_range(total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous, balanced [begin, end) slice of `total` items for `rank` of `world`."""
    base, rem = divmod(total, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


_COLL_CACHE: dict = {}


def _cached(key, shape, dtype, device, zero=False):
    """Buffers of the collectives are allocated once per (role, shape, dtype, device) and reused by every later call."""
    k = (key, tuple(shape), dtype, str(device))
    t = _COLL_CACHE.get(k)
    if t is None:
        t = (torch.zeros if zero else torch.empty)(tuple(shape), dtype=dtype, device=device)
        _COLL_CACHE[k] = t
    return t


def allgather_shards(local: torch.Tensor, total: int, rank: int, world: int, group=None, tag=None) -> torch.Tensor:
    """Every rank holds items shard_range(total, rank, world) along dim 0; returns all `total`
    items on every rank (one padded all_gather into a preallocated buffer; NCCL on CUDA, gloo on CPU tensors).
    The result may BE that buffer (one per `tag`, shape and dtype): it is overwritten by the next call with the same tag."""
    if world == 1:
        return local.contiguous()
    import torch.distributed as dist
    per = (total + world - 1) // world
    tail = tuple(local.shape[1:])
    pad = _cached("ag_in", (per,) + tail, local.dtype, local.device, zero=True)
    pad[: local.shape[0]] = local
    full = _cached(("ag_out", tag), (world * per,) + tail, local.dtype, local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(full, pad, group=group)
    else:                                            # gloo: list form
        dist.all_gather(list(full.view((world, per) + tail).unbind(0)), pad, group=group)
    if total == world * per:
        return full
    parts = full.view((world, per) + tail)
    out = []
    for r in range(world):
        a, b = shard_range(total, r, world)
        out.append(parts[r][: b - a])
    return torch.cat(out).contiguous()


def gather_bands(band: torch.Tensor, total_rows: int, rank: int, world: int, group=None, dst: int = 0, tag=None):
    """Row bands shard_range(total_rows, r, world) -> the full [total_rows, ...] tensor on group rank
    `dst` (None elsewhere): the final mask gather.  Receive buffers are preallocated views of one tensor per `tag`:
    the returned tensor IS that buffer when the bands divide evenly, so results that must stay alive side by side
    (the masks of one segment() call) need distinct tags; a later call with the same tag overwrites it."""
    if world == 1:
        return band
    import torch.distributed as dist
    per = (total_rows + world - 1) // world
    tail = tuple(band.shape[1:])
    if band.shape[0] == per:
        pad = band.contiguous()
    else:
        pad = _cached("gb_in", (per,) + tail, band.dtype, band.device, zero=True)
        pad[: band.shape[0]] = band
    full = _cached(("gb_out", id(group), tag), (world * per,) + tail, band.dtype, band.device) if rank == dst else None
    buf = list(full.view((world, per) + tail).unbind(0)) if rank == dst else None
    gdst = dist.get_global_rank(group, dst) if group is not None else dst
    dist.gather(pad, buf, dst=gdst, group=group)
    if rank != dst:
        return None
    if total_rows == world * per:
        return full
    out = []
    for r in range(world):
        a, b = shard_range(total_rows, r, world)
        out.append(buf[r][: b - a])
    return torch.cat(out)


def allreduce_minmax(minmax_ord: torch.Tensor, group=None) -> None:
    """minmax_ord int32 [2] (order-preserving keys): element 0 reduces with MIN, element 1 with MAX."""
    import torch.distributed as dist
    dist.all_reduce(minmax_ord[0:1], op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(minmax_ord[1:2], op=dist.ReduceOp.MAX, group=group)


def shared_pinned_u8(path: str, shape, create: bool) -> torch.Tensor:
    """uint8 HOST tensor backed by a shared file mapping (put `path` under /dev/shm) and page-locked with cudaHostRegister, so
    that several single-GPU processes can each copy their band of a mask device -> host into ONE image, in parallel over their
    own PCIe links.  The creator passes create=True before the others open it; unlink the file when done."""
    numel = 1
    for d in shape:
        numel *= int(d)
    if create:
        with open(path, "wb") as f:
            f.truncate(numel)
    t = torch.from_file(path, shared=True, size=numel, dtype=torch.uint8)
    rc = torch.cuda.cudart().cudaHostRegister(t.data_ptr(), numel, 0)
    if int(rc) != 0:
        raise _lib.VitocmError(f"cudaHostRegister failed with {rc}")
    return t.view(*shape)


class MosaicSegmenter:
    """Sliding-window white-matter segmentation of a gray mosaic (SSS/sw_processing.py:223-262).

    model: vitocm VisionTransformer (patch 8); window/stride: crop geometry (reference default
    384/128; BASELINE configs use 224/112); tile_batch: most tiles per engine call (the shard is cut into equal calls); group: optional
    torch.distributed process group (NCCL) to shard over -- None = single GPU; ingest: "direct" = the
    patch embedding reads its pixels straight out of the uint8 mosaic, "crops" = fp32 crops are cut first
    (vitocm_extract_tiles); both give the same bits."""

    def __init__(self, model, window=384, stride=128, tile_batch=512, group=None, ingest="direct"):
        if ingest not in ("direct", "crops"):
            raise ValueError("ingest must be 'direct' (tiles read out of the mosaic by the patch embedding) or 'crops' (materialised fp32 crops)")
        self.ingest = ingest
        self.model = model
        self.window, self.stride, self.tile_batch = int(window), int(stride), int(tile_batch)
        self.group = group
        if group is not None:
            import torch.distributed as dist
            self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        else:
            self.rank, self.world = 0, 1
        self.patch = model.patch_embed.patch_size
        if self.window % self.patch:
            raise ValueError("window must be a multiple of the patch size")

    @torch.no_grad()
    def lowres_maps(self, mosaic, t0: int, t1: int) -> torch.Tensor:
        """Per-tile normalised low-res maps [t1-t0, h, w] for tiles t0..t1-1 (row-major) of the mosaic's ny x nx window grid
        (mosaic_grid).  mosaic: uint8 CUDA tensor, or a tuple (device address of row 0, height, width, pitch, device) for a band
        buffer addressed by absolute rows."""
        lib = _lib.load_library()
        W, S = self.window, self.stride
        C = 1          # the mosaic is gray: one channel per tile and the channel-folded patch filter (gray fast path)
        if isinstance(mosaic, tuple):
            mos_ptr, mos_h, mos_w, pitch, dev = mosaic
        else:
            mos_ptr, mos_h, mos_w, pitch, dev = mosaic.data_ptr(), mosaic.shape[0], mosaic.shape[1], mosaic.stride(0), mosaic.device
        grid = (grid_size(mos_h, S), grid_size(mos_w, S))
        lh = W // self.patch
        out = torch.empty(max(t1 - t0, 0), lh * lh, dtype=torch.float32, device=dev)
        direct = self.ingest == "direct" and self.model.in_chans > 1
        xbuf = None if direct else torch.empty(self.tile_batch, C, W, W, dtype=torch.float32, device=dev)
        # engine calls of (nearly) equal size, none larger than tile_batch: every kernel is a persistent grid over equal work
        # items, so a short last call would run its partial wave at the cost of a full one
        calls = max(1, -(-(t1 - t0) // self.tile_batch))
        bounds = [t0 + (t1 - t0) * i // calls for i in range(calls + 1)]
        for a, b in zip(bounds[:-1], bounds[1:]):
            if direct:   # the patch-embedding producer reads the uint8 mosaic itself: no crop is materialised
                rows = self.model.cls_attention_rows_mosaic((mos_ptr, mos_h, mos_w, pitch, dev), grid, W, S, a, b - a)
            else:
                x = xbuf[: b - a]
                check(lib.vitocm_extract_tiles_grid(mos_ptr, mos_h, mos_w, pitch, *grid, W, S, a, b - a, C, ptr(x), cur_stream()))
                rows = self.model.cls_attention_rows(x)
            out[a - t0:b - t0] = head_mean_maps(rows, per_tile_minmax255=True)
        return out.view(-1, lh, lh)

    def mosaic_rows_needed(self, height: int, width: int | None = None) -> tuple[int, int]:
        """Rows [r0, r1) of a height x width mosaic (width defaults to height) that this rank reads: the windows of its tile
        shard and its band of output rows."""
        W, S = self.window, self.stride
        (ny, nx), (Ey, _) = mosaic_grid(height, height if width is None else width, S, W)
        T = ny * nx
        t0, t1 = shard_range(T, self.rank, self.world)
        y0, y1 = shard_range(Ey, self.rank, self.world)
        r0, r1 = y0, y1
        if t1 > t0:
            r0 = min(r0, (t0 // nx) * S)
            r1 = max(r1, ((t1 - 1) // nx) * S + W)
        return max(r0, 0), min(r1, height)

    @torch.no_grad()
    def segment(self, mosaic: torch.Tensor, want=("th", "th3"), gather: bool = True, host_out: dict | None = None):
        """mosaic: uint8 gray [H, W] (any aspect ratio), a CUDA tensor or a HOST tensor (pinned for an asynchronous copy).  Its
        ny x nx window grid and Ey x Ex stitched extent are mosaic_grid(H, W, stride, window): rows of windows come from the
        height, columns from the width.  A host mosaic is uploaded band-wise: every rank copies only the rows its own windows and
        output rows touch (mosaic_rows_needed), so R ranks move ~1/R of the image each over their own PCIe link instead of R
        whole copies.  host_out: optional dict name -> uint8 HOST tensor [Ey, Ex] (pinned; for several ranks a shared mapping,
        see shared_pinned_u8): every rank copies its band of each mask straight into rows [y0, y1) of it -- the final "gather"
        then happens in host memory, in parallel, and the NCCL gather to rank 0 is skipped unless gather=True.
        Returns dict with the masks of this rank's row band (and, on rank 0 with gather=True, the full [Ey, Ex] masks),
        thresholds, min/max, lowres; grid_shape = (ny, nx) and extent_shape = (Ey, Ex); grid / extent = n / E for a square
        mosaic and the (ny, nx) / (Ey, Ex) pairs otherwise."""
        if mosaic.dtype != torch.uint8 or mosaic.dim() != 2:
            raise ValueError("mosaic must be a 2-D uint8 gray tensor")
        lib = _lib.load_library()
        W, S = self.window, self.stride
        H, Wd = int(mosaic.shape[0]), int(mosaic.shape[1])
        (ny, nx), (Ey, Ex) = mosaic_grid(H, Wd, S, W)
        if ny < 1 or nx < 1:
            raise ValueError(f"mosaic {H} x {Wd} smaller than one window along an axis (window {W}, stride {S})")
        T = ny * nx
        lh = W // self.patch
        dev = _dev() if not mosaic.is_cuda else mosaic.device
        if mosaic.is_cuda:
            mos_ptr, pitch = mosaic.data_ptr(), mosaic.stride(0)
            mos_keep = mosaic
        else:
            if mosaic.stride(1) != 1:
                raise ValueError("host mosaic must have unit column stride")
            r0, r1 = self.mosaic_rows_needed(H, Wd)
            mos_keep = _cached("mosaic_band", (max(r1 - r0, 1), Wd), torch.uint8, dev)
            mos_keep[: r1 - r0].copy_(mosaic[r0:r1], non_blocking=True)
            pitch = Wd
            mos_ptr = mos_keep.data_ptr() - r0 * pitch      # absolute-row addressing: rows outside [r0, r1) are never read
        wtab = _wtab(W, S, dev)
        # 1. ViT on this rank's tiles
        t0, t1 = shard_range(T, self.rank, self.world)
        mine = self.lowres_maps((mos_ptr, H, Wd, pitch, dev), t0, t1)
        lowres = allgather_shards(mine, T, self.rank, self.world, self.group, tag=id(self))
        # 2. this rank's band of output rows
        y0, y1 = shard_range(Ey, self.rank, self.world)
        gray_band = torch.empty(max(y1 - y0, 1), Ex, dtype=torch.uint8, device=dev)    # this rank's rows only
        gray_base = gray_band.data_ptr() - y0 * Ex                                      # absolute-row addressing (see _threshold_device)
        check(lib.vitocm_stitch_gray_grid(mos_ptr, H, Wd, pitch, ny, nx, W, S, ptr(wtab), y0, y1, gray_base, cur_stream()))
        masks, thr, minmax, hists = _threshold_device(lib, lowres, (ny, nx, W, S, lh, lh), wtab, None, None, y0, y1,
                                                      group=self.group if self.world > 1 else None, want=want, gray_base=gray_base)
        square = ny == nx
        out = dict(band=(y0, y1), thresholds=thr, minmax_ord=minmax, hists=hists, lowres=lowres,
                   extent=Ey if square else (Ey, Ex), grid=ny if square else (ny, nx), extent_shape=(Ey, Ex), grid_shape=(ny, nx))
        out.update({k + "_band": v for k, v in masks.items()})
        if host_out is not None:
            for k, v in masks.items():
                if k in host_out and y1 > y0:
                    host_out[k][y0:y1].copy_(v, non_blocking=True)
        # 3. final mask gather on rank 0
        if self.world > 1 and gather:
            for k, v in masks.items():
                # receive buffers belong to this segmenter and this mask: the returned full masks stay valid until THIS
                # segmenter's next segment() call
                full = gather_bands(v, Ey, self.rank, self.world, self.group, dst=0, tag=(id(self), k))
                if full is not None:
                    out[k] = full
        elif self.world == 1:
            out.update(masks)
        return out

    @torch.no_grad()
    def stitched_map(self, lowres: torch.Tensor, grid=None) -> torch.Tensor:
        """The full stitched attention map [Ey, Ex] fp32 (:259) from low-res maps (for inspection / tests).  grid: (ny, nx) of a
        rectangular mosaic (segment()'s grid_shape); None infers a square n x n grid from the tile count."""
        lib = _lib.load_library()
        W, S = self.window, self.stride
        if grid is None:
            n = int(round(lowres.shape[0] ** 0.5))
            ny = nx = n
        else:
            ny, nx = int(grid[0]), int(grid[1])
            if ny * nx != lowres.shape[0]:
                raise ValueError(f"stitched_map: {lowres.shape[0]} low-res maps for a {ny} x {nx} grid")
        Ey, Ex = (ny - 1) * S + W, (nx - 1) * S + W
        lh = lowres.shape[-1]
        wtab = _wtab(W, S, lowres.device)
        minmax = torch.empty(2, dtype=torch.int32, device=lowres.device)
        out = torch.empty(Ey, Ex, dtype=torch.float32, device=lowres.device)
        check(lib.vitocm_minmax_init(ptr(minmax), cur_stream()))
        check(lib.vitocm_stitch_minmax_grid(ptr(lowres.contiguous()), ny, nx, W, S, lh, lh, ptr(wtab), 0, Ey, ptr(minmax), ptr(out),
                                            None, cur_stream()))
        return out
