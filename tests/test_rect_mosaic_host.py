"""CPU: rectangular mosaics -- the ny x nx grid oracle against the reference-pinned square one and against the separable
two-axis statement of the stitch, the band arithmetic of the sharded path (gloo, world_size 2), the grid entry points of the
C ABI and their argument checks, and the touched mosaic kernels as ptxas builds them for sm_100a."""
import ctypes as C
import os
import re
import shutil
import socket
import subprocess
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch

import vitocm_b200 as vob
from conftest import ROOT, load_golden
from oracle import post_oracle as PO
from rect_mosaic_oracle import (concat_crops_blend_grid, grid_of, mosaic_segment_grid, separable_stitch,
                                sliding_window_grid)

CSRC = os.path.join(ROOT, "vit-ocm-wmsegmentation_b200", "csrc")


# ----------------------------------------------------------------------------- oracle
@pytest.mark.parametrize("name,W,S,n", [("w32s16n4", 32, 16, 4), ("w48s16n3", 48, 16, 3), ("w24s8n5", 24, 8, 5), ("w32s16n1", 32, 16, 1)])
def test_grid_oracle_reduces_to_the_reference_pinned_square_one(name, W, S, n):
    g = load_golden("stitch.npz")
    tiles = list(g[name + "/tiles"])
    out = concat_crops_blend_grid(tiles, n, n, S, W)
    assert out.dtype == np.float32 and np.array_equal(out, g[name + "/out"])
    assert np.array_equal(out, PO.concat_crops_blend(tiles, S, W))
    if name + "/img" in g:
        img = g[name + "/img"]
        for im in (img, np.stack([img] * 3, -1)):
            got, want = sliding_window_grid(im, S, W), PO.sliding_window(im, S, W)
            assert len(got) == len(want) == n * n and all(np.array_equal(a, b) for a, b in zip(got, want))
        gray = concat_crops_blend_grid(sliding_window_grid(img, S, W), n, n, S, W)
        assert np.array_equal(gray, g[name + "/gray_stitched"])


def test_mosaic_segment_grid_equals_mosaic_segment_on_a_square():
    rng = np.random.RandomState(4)
    size, W, S = 100, 32, 16
    n = vob.grid_size(size, S)
    rows = rng.rand(n * n, 2, (W // 8) ** 2 + 1).astype(np.float32)
    mosaic = rng.randint(0, 256, (size, size)).astype(np.uint8)
    a_st, a_th, a_gray = mosaic_segment_grid(rows, mosaic, S, W)
    b_st, b_th, b_gray = PO.mosaic_segment(rows, mosaic, S, W)
    assert np.array_equal(a_st, b_st) and np.array_equal(a_gray, b_gray)
    assert all(np.array_equal(x, y) for x, y in zip(a_th, b_th))


@pytest.mark.parametrize("ny,nx", [(3, 5), (5, 2), (1, 4), (4, 1), (1, 1)])
@pytest.mark.parametrize("W,S", [(32, 16), (48, 16), (24, 8)])
def test_rectangular_blend_equals_the_separable_two_axis_profiles(ny, nx, W, S):
    """Tall, wide, single-row and single-column grids: the sequential blend of float64 crops equals the separable statement to
    float64 rounding, and that of float32 crops (a rounding at every seam) to float32 rounding."""
    rng = np.random.RandomState(ny * 10 + nx)
    crops = [rng.rand(W, W) * 255.0 for _ in range(ny * nx)]
    ref = separable_stitch(crops, ny, nx, S, W)
    Ey, Ex = (ny - 1) * S + W, (nx - 1) * S + W
    got64 = concat_crops_blend_grid(crops, ny, nx, S, W)
    assert got64.shape == (Ey, Ex) and np.abs(got64 - ref).max() <= 1e-9
    got32 = concat_crops_blend_grid([c.astype(np.float32) for c in crops], ny, nx, S, W)
    assert got32.dtype == np.float32 and np.abs(got32 - ref).max() <= 255.0 * 4e-7


def test_sliding_window_grid_walks_rows_over_the_height():
    rng = np.random.RandomState(2)
    img = rng.randint(0, 256, (70, 131)).astype(np.uint8)
    (ny, nx), _ = grid_of(70, 131, 16, 32)
    crops = sliding_window_grid(img, 16, 32)
    assert (ny, nx) == (vob.grid_size(70, 16), vob.grid_size(131, 16)) == vob.mosaic_grid(70, 131, 16, 32)[0]
    assert len(crops) == ny * nx
    for t, c in enumerate(crops):
        y, x = (t // nx) * 16, (t % nx) * 16
        want = np.zeros((32, 32), np.uint8)
        part = img[y:y + 32, x:x + 32]
        want[: part.shape[0], : part.shape[1]] = part
        assert np.array_equal(c, want), t


# ----------------------------------------------------------------------------- band arithmetic
def _segmenter(rank, world, window=224, stride=112):
    seg = vob.MosaicSegmenter(NS(patch_embed=NS(patch_size=8)), window=window, stride=stride)
    seg.rank, seg.world = rank, world
    return seg


def _check_bands(H, Wd, window, stride, world):
    (ny, nx), (Ey, Ex) = vob.mosaic_grid(H, Wd, stride, window)
    covered = np.zeros(Ey, np.int32)
    for rank in range(world):
        seg = _segmenter(rank, world, window, stride)
        r0, r1 = seg.mosaic_rows_needed(H, Wd)
        assert 0 <= r0 <= r1 <= H
        t0, t1 = vob.shard_range(ny * nx, rank, world)
        for t in range(t0, t1):
            oy = (t // nx) * stride
            assert r0 <= oy and min(oy + window, H) <= r1, (H, Wd, world, rank, t)
        y0, y1 = vob.shard_range(Ey, rank, world)
        covered[y0:y1] += 1
        if y1 > y0:        # the stitched gray image of the band reads the mosaic rows of the band
            assert r0 <= min(y0, H) and min(y1, H) <= r1
    assert (covered == 1).all()


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_mosaic_rows_needed_for_rectangles(world):
    for H, Wd, window, stride in ((3024, 5712, 224, 112), (5712, 3024, 224, 112), (4096, 8192, 224, 112), (112, 176, 32, 16),
                                  (176, 100, 48, 16), (128, 48, 32, 16), (48, 128, 32, 16), (100, 100, 32, 16)):
        _check_bands(H, Wd, window, stride, world)
    # the square form keeps its meaning
    seg = _segmenter(0, 2)
    assert seg.mosaic_rows_needed(4096) == seg.mosaic_rows_needed(4096, 4096)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gloo_worker(rank, world, port, tmp):
    import torch.distributed as dist
    import vitocm_b200 as v
    from vitocm_b200 import sw_processing as sw
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        H, Wd, window, stride = 176, 100, 48, 16
        (ny, nx), (Ey, Ex) = v.mosaic_grid(H, Wd, stride, window)
        seg = v.MosaicSegmenter(NS(patch_embed=NS(patch_size=8)), window=window, stride=stride, group=dist.group.WORLD)
        assert (seg.rank, seg.world) == (rank, world)
        r0, r1 = seg.mosaic_rows_needed(H, Wd)
        t0, t1 = v.shard_range(ny * nx, rank, world)
        assert all(r0 <= (t // nx) * stride and min((t // nx) * stride + window, H) <= r1 for t in range(t0, t1))
        g = torch.Generator().manual_seed(0)
        maps = torch.rand(ny * nx, 6, 6, generator=g)
        assert torch.equal(sw.allgather_shards(maps[t0:t1].clone(), ny * nx, rank, world), maps)
        mask = (torch.rand(Ey, Ex, generator=g) > 0.5).to(torch.uint8)
        y0, y1 = v.shard_range(Ey, rank, world)
        got = sw.gather_bands(mask[y0:y1].clone(), Ey, rank, world, dst=0, tag="rect")
        if rank == 0:
            assert torch.equal(got, mask)
        else:
            assert got is None
        open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_rectangular_bands_gloo_world2(tmp_path):
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(tmp_path / f"ok{r}") for r in range(world))


# ----------------------------------------------------------------------------- C ABI
GRID_FORMS = {   # grid form -> its n-form: one argument more (n -> ny, nx), otherwise the same
    "vitocm_forward_cls_attn_mosaic_grid": "vitocm_forward_cls_attn_mosaic",
    "vitocm_extract_tiles_grid": "vitocm_extract_tiles",
    "vitocm_stitch_gray_grid": "vitocm_stitch_gray",
    "vitocm_stitch_minmax_grid": "vitocm_stitch_minmax",
    "vitocm_stitch_hist_grid": "vitocm_stitch_hist",
    "vitocm_stitch_mask_grid": "vitocm_stitch_mask",
    "vitocm_stitch_result_grid": "vitocm_stitch_result",
    "vitocm_concat_crops_grid_f32": "vitocm_concat_crops_f32",
    "vitocm_concat_crops_grid_u8": "vitocm_concat_crops_u8",
}


def test_grid_entry_points_load_with_their_argtypes(lib):
    assert lib.vitocm_version() == 100
    for grid, nform in GRID_FORMS.items():
        fn, fn_n = getattr(lib, grid), getattr(lib, nform)
        ga, na = list(fn.argtypes), list(fn_n.argtypes)
        assert len(ga) == len(na) + 1, grid
        # the grid form takes `ny, nx` where the n-form takes its int `n`; every other argument is unchanged
        assert any(ga[k] is C.c_int and ga[k + 1] is C.c_int and ga[:k] + ga[k + 1:] == na for k in range(len(na))), grid


def _err(lib, rc):
    assert rc != 0
    return lib.vitocm_last_error().decode()


def test_bad_grids_are_refused_before_any_launch(lib):
    """Argument errors come back through vitocm_last_error without any device work (this runs without a GPU, where a launch
    would report a CUDA error instead)."""
    N = None
    one = 1
    for ny, nx in ((0, 3), (3, 0), (-1, 2)):
        assert "bad sliding-window geometry" in _err(lib, lib.vitocm_stitch_gray_grid(one, 10, 10, 10, ny, nx, 32, 16, N, 0, 1, one, N))
        assert "bad sliding-window geometry" in _err(lib, lib.vitocm_stitch_minmax_grid(N, ny, nx, 32, 16, 4, 4, N, 0, 1, one, N, one, N))
        assert "bad sliding-window geometry" in _err(lib, lib.vitocm_concat_crops_grid_f32(one, ny, nx, 32, 16, N, one, N))
        assert "bad window grid" in _err(lib, lib.vitocm_extract_tiles_grid(one, 10, 10, 10, ny, nx, 32, 16, 0, 1, 1, one, N))
        assert "bad window grid" in _err(lib, lib.vitocm_forward_cls_attn_mosaic_grid(N, one, 10, 10, 10, ny, nx, 32, 16, 0, 1, one,
                                                                                       one, one, 0, 1, N))
    # windows beyond the grid
    assert "bad window grid" in _err(lib, lib.vitocm_extract_tiles_grid(one, 10, 10, 10, 2, 3, 32, 16, 4, 3, 1, one, N))
    assert "bad window grid" in _err(lib, lib.vitocm_forward_cls_attn_mosaic_grid(N, one, 10, 10, 10, 3, 2, 32, 16, 0, 7, one, one,
                                                                                   one, 0, 1, N))
    # a band outside [0, Ey): Ey = (2 - 1) * 16 + 32 = 48 although Ex = 96
    for fn in (lambda y1: lib.vitocm_stitch_hist_grid(N, 2, 5, 32, 16, 4, 4, N, one, one, 0, y1, one, N, N),
               lambda y1: lib.vitocm_stitch_mask_grid(N, 2, 5, 32, 16, 4, 4, N, one, one, one, 0, y1, N, N, N, N, N),
               lambda y1: lib.vitocm_stitch_result_grid(N, 2, 5, 32, 16, 4, 4, N, one, one, 0, y1, N, N, N, N)):
        assert "bad row band [0,49) for extent 48" in _err(lib, fn(49))
    # too much overlap, window not wider than the stride
    assert "at most four windows" in _err(lib, lib.vitocm_concat_crops_grid_u8(one, 2, 3, 80, 16, 1, N, one, N))
    assert "bad sliding-window geometry" in _err(lib, lib.vitocm_concat_crops_grid_u8(one, 2, 3, 16, 16, 1, N, one, N))
    # and the n-forms are the grid forms with ny = nx = n
    assert "bad sliding-window geometry 0x0" in _err(lib, lib.vitocm_stitch_gray(one, 10, 10, 10, 0, 32, 16, N, 0, 1, one, N))


def test_rectangular_segment_input_checks_on_the_host():
    seg = _segmenter(0, 1, 32, 16)
    with pytest.raises(ValueError, match="smaller than one window"):
        seg.segment(torch.zeros(200, 32, dtype=torch.uint8))
    with pytest.raises(ValueError, match="2-D uint8"):
        seg.segment(torch.zeros(2, 64, 64, dtype=torch.uint8))


# ----------------------------------------------------------------------------- kernels
_UNIT = """
#include "post_kernels.cuh"
namespace vitocm {
void* const mosaic_kernels[] = {
  reinterpret_cast<void*>(extract_tiles_kernel),
  reinterpret_cast<void*>(stitch_gray_kernel<1>), reinterpret_cast<void*>(stitch_gray_kernel<4>),
  reinterpret_cast<void*>(stitch_gray_strip_kernel<1, 2>), reinterpret_cast<void*>(stitch_gray_strip_kernel<1, 4>),
  reinterpret_cast<void*>(stitch_gray_strip_kernel<4, 2>), reinterpret_cast<void*>(stitch_gray_strip_kernel<4, 4>),
  reinterpret_cast<void*>(stitch_minmax_kernel<1>), reinterpret_cast<void*>(stitch_minmax_kernel<4>),
  reinterpret_cast<void*>(stitch_strip_kernel<2>), reinterpret_cast<void*>(stitch_strip_kernel<4>),
  reinterpret_cast<void*>(stitch_hist_kernel<1>), reinterpret_cast<void*>(stitch_hist_kernel<4>),
  reinterpret_cast<void*>(stitch_mask_kernel<1>), reinterpret_cast<void*>(stitch_mask_kernel<4>),
  reinterpret_cast<void*>(stitch_result_kernel<1>), reinterpret_cast<void*>(stitch_result_kernel<4>),
  reinterpret_cast<void*>(concat_crops_f32_kernel), reinterpret_cast<void*>(concat_crops_u8_kernel),
};
}
"""


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    pytest.skip("nvcc not available")


def test_grid_mosaic_kernels_build_for_sm100a(tmp_path):
    """Every mosaic kernel compiles for sm_100a.  Spills stay where they were before the kernels took ny x nx grids: none, except
    the 4-byte spill of the four-window column-strip stitch."""
    nvcc = _nvcc()
    src = tmp_path / "mosaic.cu"
    src.write_text(_UNIT)
    res = subprocess.run([nvcc, "-cubin", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", CSRC, "-o", str(tmp_path / "mosaic.cubin"), str(src)], capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    log = res.stdout + res.stderr
    spills = {name: int(st) + int(ld) for name, st, ld in
              re.findall(r"Function properties for (\S+)\n\s+\d+ bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)}
    kernels = [k for k in spills if re.search(r"stitch_|concat_crops_(f32|u8)_kernel|extract_tiles_kernel", k)]
    assert len(kernels) == 19, kernels
    for k in kernels:
        allowed = 8 if k.startswith("_ZN6vitocm19stitch_strip_kernelILi4E") else 0
        assert spills[k] <= allowed, (k, spills[k])
