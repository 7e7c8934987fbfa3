"""Oracle for rectangular mosaics (test infrastructure): the sliding window, the ramp-blended concat_crops and the mosaic
driver of oracle/post_oracle.py on an ny x nx window grid, with rows of windows over the height and columns over the width.

The reference cannot run a rectangle (its concat_crops takes n = sqrt(len(crops)) and its sliding_window swaps PIL's (W, H)),
so these are the reference's loops with the two axes given their own counts; every arithmetic step (the float64 ramp, the
dtype of the running image, the per-tile normalisation, the resize pair, threshold_sw) is post_oracle's.  On a square grid
they reduce to post_oracle's reference-pinned sliding_window / concat_crops_blend / mosaic_segment
(tests/test_rect_mosaic_host.py checks this)."""
from __future__ import annotations

import numpy as np

from oracle import post_oracle as PO


def grid_of(height: int, width: int, stride: int, window: int):
    """((ny, nx), (Ey, Ex)) of a height x width mosaic."""
    ny, nx = len(PO.sliding_window_origins(height, stride)), len(PO.sliding_window_origins(width, stride))
    return (ny, nx), ((ny - 1) * stride + window, (nx - 1) * stride + window)


def sliding_window_grid(image: np.ndarray, stride: int, window: int) -> list[np.ndarray]:
    """Row-major windows of an [H, W(, C)] image: origins range(0, H - 2S, S) down the rows, range(0, W - 2S, S) across;
    zero padded beyond the image like PIL's crop."""
    image = np.asarray(image)
    hgt, wid = image.shape[0], image.shape[1]
    crops = []
    for y in PO.sliding_window_origins(hgt, stride):
        for x in PO.sliding_window_origins(wid, stride):
            win = np.zeros((window, window) + image.shape[2:], dtype=image.dtype)
            ys, xs = min(y + window, hgt), min(x + window, wid)
            if ys > y and xs > x:
                win[: ys - y, : xs - x] = image[y:ys, x:xs]
            crops.append(win)
    return crops


def concat_crops_blend_grid(crops: list[np.ndarray], ny: int, nx: int, stride: int, window_size: int) -> np.ndarray:
    """SSS/sw_processing.py:113-134 on ny strips of nx crops: blend along x inside each strip, then along y across strips."""
    step = window_size - stride
    vertical = None
    for i in range(ny):
        horizontal = crops[i * nx]
        for j in range(1, nx):
            right = crops[i * nx + j]
            overlap = PO._blend_h(horizontal[:, -step:], right[:, :-stride])
            horizontal = np.concatenate((horizontal[:, :-step], overlap, right[:, -stride:]), axis=1)
        if i == 0:
            vertical = horizontal
        else:
            top = PO._blend_v(vertical[-step:, :], horizontal[:-stride, :])
            vertical = np.concatenate((vertical[:-step, :], top, horizontal[-stride:, :]), axis=0)
    return vertical


def blend_profiles_grid(ny: int, nx: int, stride: int, window_size: int):
    """The two-axis separable statement of the float stitch: out(y, x) = sum_ij Py[i, y] Px[j, x] tile_ij(y - iS, x - jS),
    Py = blend_profiles(ny) [ny, Ey] and Px = blend_profiles(nx) [nx, Ex] (float64)."""
    return PO.blend_profiles(ny, stride, window_size), PO.blend_profiles(nx, stride, window_size)


def separable_stitch(crops: list[np.ndarray], ny: int, nx: int, stride: int, window_size: int) -> np.ndarray:
    """Stitch a 2-D float grid of crops through blend_profiles_grid, in float64."""
    Py, Px = blend_profiles_grid(ny, nx, stride, window_size)
    out = np.zeros((Py.shape[1], Px.shape[1]), dtype=np.float64)
    for i in range(ny):
        for j in range(nx):
            y0, x0 = i * stride, j * stride
            wy = Py[i, y0:y0 + window_size][:, None]
            wx = Px[j, x0:x0 + window_size][None, :]
            out[y0:y0 + window_size, x0:x0 + window_size] += wy * wx * np.asarray(crops[i * nx + j], dtype=np.float64)
    return out


def mosaic_segment_grid(cls_rows_all: np.ndarray, mosaic_u8: np.ndarray, stride: int, window: int, patch_size: int = 8):
    """sw_processing.py:223-262 on a rectangular mosaic.  cls_rows_all: [ny*nx, H, N] for the row-major windows of
    sliding_window_grid; mosaic_u8: gray [H, W].  Returns (stitched float32 [Ey, Ex], threshold_sw tuple, stitched gray)."""
    (ny, nx), _ = grid_of(mosaic_u8.shape[0], mosaic_u8.shape[1], stride, window)
    maps = [PO.sw_tile_map(cls_rows_all[t], window, patch_size) for t in range(ny * nx)]
    stitched = concat_crops_blend_grid(maps, ny, nx, stride, window)
    crops = sliding_window_grid(mosaic_u8, stride, window)
    gray = concat_crops_blend_grid(crops, ny, nx, stride, window)
    return stitched, PO.threshold_sw(gray, stitched), gray
