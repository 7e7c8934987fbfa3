"""GPU (B200): rectangular mosaics through MosaicSegmenter and the grid entry points of the C ABI.  The ViT stage is held to the
tolerance of the square pipeline test; everything after it, fed the GPU's own CLS rows, must equal the ny x nx grid oracle bit
for bit.  Square mosaics through the grid forms must equal the n-forms bit for bit."""
import numpy as np
import pytest
import torch

import vitocm_b200 as vob
import rect_mosaic_oracle as RO
from gpu_util import build_model
from oracle import post_oracle as PO
from oracle import vit_oracle as VO
from vitocm_b200 import sw_processing as sw
from vitocm_b200 import synthetic as syn
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu


def _rect_mosaic(H, Wd, seed):
    return np.ascontiguousarray(VO.synthetic_mosaic_u8(max(H, Wd), seed=seed)[:H, :Wd])


def _tiny(W, precision="fp32"):
    tiny = VO.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=8, img_size=W)
    sd = VO.randomize_affine(VO.init_state_dict(tiny, seed=21), seed=22)
    return tiny, sd, build_model(tiny, sd, precision, chunk_tiles=5)


@pytest.mark.parametrize("H,Wd,W,S", [(112, 176, 32, 16), (176, 100, 32, 16), (128, 48, 32, 16),
                                      (112, 176, 48, 16), (176, 100, 48, 16), (128, 48, 48, 16),
                                      (48, 160, 32, 16), (40, 100, 48, 16)])
def test_rectangular_pipeline_vs_grid_oracle(H, Wd, W, S):
    """Tall and wide mosaics, W % S != 0 (48 / 16 is 3 windows per point, 32 / 16 two), ragged edges (100, 176 are not window
    multiples), one column of windows (width 48) and one row (heights 48 and 40)."""
    tiny, sd, m = _tiny(W)
    mosaic = _rect_mosaic(H, Wd, seed=77)
    (ny, nx), (Ey, Ex) = RO.grid_of(H, Wd, S, W)
    assert (ny == 1) == (H <= 48) and (nx == 1) == (Wd == 48)
    seg = vob.MosaicSegmenter(m, window=W, stride=S, tile_batch=7)
    out = seg.segment(torch.from_numpy(mosaic).cuda(), want=("th", "th2", "th3"))
    assert out["grid_shape"] == (ny, nx) and out["extent_shape"] == (Ey, Ex)
    assert out["grid"] == (ny if ny == nx else (ny, nx)) and out["extent"] == (Ey if ny == nx else (Ey, Ex))
    # ViT stage vs oracle
    crops = RO.sliding_window_grid(mosaic, S, W)
    xs = torch.from_numpy(np.stack(crops)).float().div(255.0).unsqueeze(1).expand(-1, 3, -1, -1).contiguous()
    rows_ref = VO.cls_attention_rows(sd, tiny, xs).numpy()
    rows_gpu = m.cls_attention_rows(xs[:, :1].contiguous().cuda()).cpu().numpy()
    assert float((np.abs(rows_gpu - rows_ref) / rows_ref).max()) <= 1e-3
    # the segmenter's own tiles are the grid's windows: its low-res maps are the head means of these rows
    low = vob.head_mean_maps(torch.from_numpy(rows_gpu).cuda(), per_tile_minmax255=True).view(ny * nx, W // 8, W // 8)
    assert torch.equal(out["lowres"], low)
    # post stage, exact, from the GPU's rows
    stitched, (th, th2, th3, _, _), gray = RO.mosaic_segment_grid(rows_gpu, mosaic, S, W, 8)
    assert stitched.shape == (Ey, Ex)
    assert np.array_equal(seg.stitched_map(out["lowres"], grid=(ny, nx)).cpu().numpy(), stitched)
    assert np.array_equal(out["th"].cpu().numpy(), th)
    assert np.array_equal(out["th2"].cpu().numpy(), th2)
    assert np.array_equal(out["th3"].cpu().numpy(), th3)
    # the stitched gray image and the function-level concat_crops on an explicit grid
    assert np.array_equal(sw.concat_crops(crops, S, W, grid=(ny, nx)), gray)
    maps = [PO.sw_tile_map(rows_gpu[t], W, 8) for t in range(ny * nx)]
    assert np.array_equal(sw.concat_crops(maps, S, W, grid=(ny, nx)), stitched)


def test_direct_ingest_equals_crops_on_a_rectangle():
    tiny, sd, m = _tiny(32, "bf16")
    lib = vob._lib.load_library()
    rng = np.random.RandomState(3)
    for H, Wd in ((101, 150), (150, 67)):
        base = rng.randint(0, 256, (H, Wd)).astype(np.uint8)
        base.flat[:256] = np.arange(256, dtype=np.uint8)
        mosaic = torch.from_numpy(base).cuda()
        ny, nx = vob.grid_size(H, 16), vob.grid_size(Wd, 16)
        T = ny * nx
        x = torch.empty(T, 1, 32, 32, device="cuda")
        check(lib.vitocm_extract_tiles_grid(mosaic.data_ptr(), H, Wd, mosaic.stride(0), ny, nx, 32, 16, 0, T, 1, ptr(x), cur_stream()))
        want_x = torch.from_numpy(np.stack(RO.sliding_window_grid(base, 16, 32))).float().div(255.0).unsqueeze(1)
        assert torch.equal(x.cpu(), want_x)
        want = m.cls_attention_rows(x)
        assert torch.equal(m.cls_attention_rows_mosaic(mosaic, (ny, nx), 32, 16, 0, T), want)
        assert torch.equal(m.cls_attention_rows_mosaic(mosaic, (ny, nx), 32, 16, 3, T - 4), want[3:T - 1])
        seg_a = vob.MosaicSegmenter(m, window=32, stride=16, tile_batch=7, ingest="direct")
        seg_b = vob.MosaicSegmenter(m, window=32, stride=16, tile_batch=7, ingest="crops")
        a, b = seg_a.segment(mosaic), seg_b.segment(mosaic)
        assert torch.equal(a["lowres"], b["lowres"]) and torch.equal(a["th"], b["th"]) and torch.equal(a["th3"], b["th3"])


def test_square_grid_forms_equal_the_n_forms_bit_for_bit():
    tiny, sd, m = _tiny(32)
    lib = vob._lib.load_library()
    size, W, S = 112, 32, 16
    n = vob.grid_size(size, S)
    E = (n - 1) * S + W
    mosaic = torch.from_numpy(VO.synthetic_mosaic_u8(size, seed=9)).cuda()
    assert torch.equal(m.cls_attention_rows_mosaic(mosaic, n, W, S, 0, n * n), m.cls_attention_rows_mosaic(mosaic, (n, n), W, S, 0, n * n))
    xa, xb = (torch.empty(n * n, 1, W, W, device="cuda") for _ in range(2))
    check(lib.vitocm_extract_tiles(ptr(mosaic), size, size, size, n, W, S, 0, n * n, 1, ptr(xa), cur_stream()))
    check(lib.vitocm_extract_tiles_grid(ptr(mosaic), size, size, size, n, n, W, S, 0, n * n, 1, ptr(xb), cur_stream()))
    assert torch.equal(xa, xb)
    low = vob.MosaicSegmenter(m, window=W, stride=S).lowres_maps(mosaic, 0, n * n).contiguous()
    wtab = sw._wtab(W, S, mosaic.device)
    res = []
    for grid in ((n,), (n, n)):
        sfx = "" if len(grid) == 1 else "_grid"
        fn = lambda name: getattr(lib, "vitocm_" + name + sfx)
        gray = torch.empty(E, E, dtype=torch.uint8, device="cuda")
        check(fn("stitch_gray")(ptr(mosaic), size, size, size, *grid, W, S, ptr(wtab), 0, E, ptr(gray), cur_stream()))
        mm = torch.empty(2, dtype=torch.int32, device="cuda")
        amap = torch.empty(E, E, device="cuda")
        check(lib.vitocm_minmax_init(ptr(mm), cur_stream()))
        check(fn("stitch_minmax")(ptr(low), *grid, W, S, 4, 4, ptr(wtab), 0, E, ptr(mm), ptr(amap), None, cur_stream()))
        hists = torch.zeros(3, 256, dtype=torch.int64, device="cuda")
        check(fn("stitch_hist")(ptr(low), *grid, W, S, 4, 4, ptr(wtab), ptr(gray), ptr(mm), 0, E, ptr(hists), None, cur_stream()))
        thr = torch.empty(3, dtype=torch.int32, device="cuda")
        check(lib.vitocm_otsu(ptr(hists), 3, ptr(thr), cur_stream()))
        masks = torch.empty(3, E, E, dtype=torch.uint8, device="cuda")
        check(fn("stitch_mask")(ptr(low), *grid, W, S, 4, 4, ptr(wtab), ptr(gray), ptr(mm), ptr(thr), 0, E, ptr(masks[0]), ptr(masks[1]),
                                ptr(masks[2]), None, cur_stream()))
        aux = torch.empty(2, E, E, dtype=torch.uint8, device="cuda")
        check(fn("stitch_result")(ptr(low), *grid, W, S, 4, 4, ptr(wtab), ptr(gray), ptr(mm), 0, E, ptr(aux[0]), ptr(aux[1]), ptr(amap),
                                  cur_stream()))
        crops = torch.rand(n * n, W, W, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
        cat = torch.empty(E, E, device="cuda")
        check(getattr(lib, "vitocm_concat_crops_f32" if len(grid) == 1 else "vitocm_concat_crops_grid_f32")(
            ptr(crops), *grid, W, S, ptr(wtab), ptr(cat), cur_stream()))
        res.append((gray, mm, amap, hists, thr, masks, aux, cat))
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_host_mosaic_and_host_out_on_a_rectangle():
    tiny, sd, m = _tiny(32)
    H, Wd = 150, 97
    mosaic = _rect_mosaic(H, Wd, seed=12)
    seg = vob.MosaicSegmenter(m, window=32, stride=16, tile_batch=7)
    dev = seg.segment(torch.from_numpy(mosaic).cuda(), want=("th", "th3"))
    Ey, Ex = dev["extent_shape"]
    host = {k: torch.zeros(Ey, Ex, dtype=torch.uint8).pin_memory() for k in ("th", "th3")}
    out = seg.segment(torch.from_numpy(mosaic).pin_memory(), want=("th", "th3"), host_out=host)
    torch.cuda.synchronize()
    assert torch.equal(out["lowres"], dev["lowres"])
    for k in ("th", "th3"):
        assert torch.equal(out[k], dev[k]) and torch.equal(host[k], dev[k].cpu())


@pytest.mark.parametrize("H,Wd", [(37, 90), (90, 37), (2, 5)])
def test_function_level_threshold_on_a_rectangle(H, Wd, tmp_path):
    from PIL import Image
    rng = np.random.RandomState(H)
    img = rng.randint(0, 256, (H, Wd)).astype(np.uint8)
    att = (rng.rand(H, Wd) * 3.0).astype(np.float32)
    got = sw.threshold(img, att, output_directory=str(tmp_path), save=True, name="case")
    th, th2, th3, result, att_u8 = PO.threshold_sw(img, att)
    assert all(np.array_equal(a, b) for a, b in zip(got, (th, th2, th3)))
    assert np.array_equal(np.array(Image.open(tmp_path / "weighted_iamge_attention.png")), result)
    assert np.array_equal(np.array(Image.open(tmp_path / "temp.png")), att_u8)
    flat = np.full((H, Wd), 0.5, np.float32)
    assert all(np.array_equal(a, b) for a, b in zip(sw.threshold(img, flat, save=False), PO.threshold_sw(img, flat)[:3]))


def test_vit_small_4096x8192_rectangle_full_size_properties():
    """ViT-S/8 at 4096 x 8192 (35 x 72 = 2520 windows of 224 at stride 112, extent 4032 x 8176), bf16: the size-independent
    properties of the square full-size test."""
    H, Wd = 4096, 8192
    mosaic = torch.from_numpy(np.concatenate([syn.synthetic_mosaic_u8(4096, seed=1), syn.synthetic_mosaic_u8(4096, seed=2)], 1)).cuda()
    torch.manual_seed(0)
    model = vob.vit_small(patch_size=8, num_classes=0, precision="bf16", chunk_tiles=175).cuda().eval()
    seg = vob.MosaicSegmenter(model, window=224, stride=112, tile_batch=175)
    out = seg.segment(mosaic, want=("th", "th2", "th3"))
    (ny, nx), (Ey, Ex) = out["grid_shape"], out["extent_shape"]
    assert (ny, nx) == (35, 72) and (Ey, Ex) == (4032, 8176) and out["grid"] == (35, 72)
    low = out["lowres"]
    assert tuple(low.shape) == (ny * nx, 28, 28) and bool(torch.isfinite(low).all())
    hists = out["hists"].cpu().numpy()
    assert hists.shape == (3, 256) and (hists.sum(1) == Ey * Ex).all()
    thr = out["thresholds"].cpu().numpy()
    assert [PO.otsu_from_hist(hists[k].astype(np.int64)) for k in range(3)] == thr.tolist()
    for key, k in (("th", 0), ("th2", 1), ("th3", 2)):
        msk = out[key]
        assert msk.dtype == torch.uint8 and tuple(msk.shape) == (Ey, Ex)
        white = int((msk == 255).sum())
        assert white + int((msk == 0).sum()) == Ey * Ex
        assert white == int(hists[k][thr[k] + 1:].sum()), key
    # 3 x 3 window neighbourhoods re-stitched by the oracle's sequential loops: interior, borders and corners
    stitched = seg.stitched_map(low, grid=(ny, nx)).cpu().numpy()
    assert stitched.shape == (Ey, Ex)
    lowc = low.cpu().numpy()
    for (i, j) in [(0, 0), (0, nx - 3), (ny - 3, 0), (ny - 3, nx - 3), (16, 40), (0, 33), (20, 0), (ny - 3, 51), (11, nx - 3)]:
        maps = [PO.resize_linear(lowc[(i + a) * nx + (j + b)], (224, 224)) for a in range(3) for b in range(3)]
        ref = PO.concat_crops_blend(maps, 112, 224)
        got = stitched[i * 112:i * 112 + 448, j * 112:j * 112 + 448]
        # rows / cols [S, 3S) of the neighbourhood are covered by no window outside it; at the mosaic's edges so are the outer ones
        y0 = 0 if i == 0 else 112
        y1 = 448 if i == ny - 3 else 336
        x0 = 0 if j == 0 else 112
        x1 = 448 if j == nx - 3 else 336
        assert np.array_equal(got[y0:y1, x0:x1], ref[y0:y1, x0:x1]), (i, j)
    # another cut of the work into engine calls and launches gives the same bits
    torch.manual_seed(0)
    model_b = vob.vit_small(patch_size=8, num_classes=0, precision="bf16", chunk_tiles=49).cuda().eval()
    out_b = vob.MosaicSegmenter(model_b, window=224, stride=112, tile_batch=64).segment(mosaic, want=("th", "th2", "th3"))
    assert torch.equal(out["lowres"], out_b["lowres"])
    for k in ("th", "th2", "th3"):
        assert torch.equal(out[k], out_b[k])
