"""GPU (B200): images of different sizes in one forward (vitocm_forward_cls_attn_varlen, VisionTransformer.cls_attention_rows_varlen,
utils.attention_masks_varlen).  A token row's arithmetic does not depend on the rows around it, and every image's rows take the kernel
route the uniform path takes for that image alone, so each image's CLS rows must equal the per-image call element for element.

The sizes cover every ragged-tail route of the attention: N = 17 (32^2, below one tile), a tail of 0 (120 x 136), <= 32 (224^2),
<= 64 (96 x 120), > 64 (96 x 160, 80^2), more than 16 full tiles (384^2), and small images whose tails pack two or four heads per
tile (56^2, 64^2)."""
import ctypes as C

import numpy as np
import pytest
import torch

import vitocm_b200 as vob
from gpu_util import attention_reference, build_model, make_engine
from oracle import vit_oracle as VO
from vitocm_b200._lib import check, cur_stream, ptr
from vitocm_b200.vision_transformer import varlen_plan

pytestmark = pytest.mark.gpu

SIZES = [(224, 224), (32, 32), (96, 160), (120, 136), (96, 120), (56, 56), (80, 80), (384, 384), (64, 64), (224, 224)]
CFGS = {
    "tiny": VO.ViTConfig(embed_dim=128, depth=3, num_heads=2, patch_size=8, img_size=64),
    "vits8": VO.ViTConfig(embed_dim=384, depth=3, num_heads=6, patch_size=8, img_size=224),
    "hd128": VO.ViTConfig(embed_dim=384, depth=3, num_heads=3, patch_size=8, img_size=224),
}
_models = {}


def _model(name, precision):
    key = (name, precision)
    if key not in _models:
        cfg = CFGS[name]
        sd = VO.randomize_affine(VO.init_state_dict(cfg, seed=31), seed=32)
        _models[key] = build_model(cfg, sd, precision, chunk_tiles=8)
    return _models[key]


def _images(sizes, chans, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.rand(chans, h, w, generator=g, device="cuda") for h, w in sizes]


@pytest.mark.parametrize("precision", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("name", ["tiny", "vits8", "hd128"])
@pytest.mark.parametrize("chans", [3, 1])
def test_varlen_rows_bit_identical_to_per_image_calls(name, precision, chans):
    m = _model(name, precision)
    ims = _images(SIZES, chans, seed=5)
    rows = m.cls_attention_rows_varlen(ims)
    assert len(rows) == len(ims)
    for i, x in enumerate(ims):
        ref = m.cls_attention_rows(x[None])[0]
        assert rows[i].shape == ref.shape
        assert torch.equal(rows[i], ref), (i, SIZES[i], (rows[i] - ref).abs().max().item())


@pytest.mark.parametrize("precision", ["fp16", "fp32"])
def test_varlen_rows_unchanged_across_chunk_budgets(precision):
    m = _model("vits8", precision)
    ims = _images(SIZES, 3, seed=6)
    ref = torch.cat([r.reshape(-1) for r in m.cls_attention_rows_varlen(ims)])
    # one chunk per image; a budget below the largest image (2305 tokens: it runs alone); everything in one chunk; a budget in between
    for budget in (1, 1000, sum(varlen_plan(SIZES, 8)["n"]), 3000):
        got = torch.cat([r.reshape(-1) for r in m.cls_attention_rows_varlen(ims, chunk_tokens=budget)])
        assert torch.equal(got, ref), budget


def test_varlen_rows_at_scale_match_per_image_calls():
    """More than 10^6 token rows (three chunks at the default budget): every persistent CTA walks many items of many images."""
    m = _model("vits8", "fp16")
    rng = np.random.default_rng(7)
    sides = [int(s) for s in rng.choice(np.arange(128, 513, 32), size=1200)]
    sizes, tok = [], 0
    for s in sides:
        sizes.append((s, s))
        tok += (s // 8) ** 2 + 1
        if tok > 1_000_000:
            break
    assert tok > 1_000_000
    ims = _images(sizes, 1, seed=8)
    rows = m.cls_attention_rows_varlen(ims)
    for i, x in enumerate(ims):
        assert torch.equal(rows[i], m.cls_attention_rows(x[None])[0]), (i, sizes[i])


def test_varlen_outputs_stay_inside_their_images():
    """NaN sentinels after the last image survive the forward and the attention; every image's CTX rows match the reference."""
    m = _model("vits8", "bf16")
    ims = _images(SIZES, 3, seed=9)
    plan = varlen_plan(SIZES, 8)
    heads, guard = m.num_heads, 4096
    out = torch.full((heads * plan["tokens"] + guard,), float("nan"), device="cuda")
    tables, pos_off, prow = {}, [], 0
    for h, w in SIZES:
        if (h, w) not in tables:
            tables[(h, w)] = (prow, m._pos_table((h // 8) * (w // 8), h, w))
            prow += tables[(h, w)][1].shape[0]
        pos_off.append(tables[(h, w)][0])
    pos = torch.cat([t for _, t in tables.values()])
    x = torch.cat([im.reshape(-1) for im in ims])
    lib = vob._lib.load_library()
    eng = m._ensure_engine()
    ws = torch.empty(int(lib.vitocm_varlen_workspace_bytes(eng, plan["cap"])), dtype=torch.uint8, device="cuda")
    hw = (C.c_int * (2 * len(SIZES)))(*[v for s in SIZES for v in s])
    po = (C.c_int * len(SIZES))(*pos_off)
    check(lib.vitocm_forward_cls_attn_varlen(eng, ptr(x), len(SIZES), 3, hw, ptr(pos), po, ptr(out), ptr(ws), ws.numel(), 0, cur_stream()))
    torch.cuda.synchronize()
    assert torch.isnan(out[heads * plan["tokens"]:]).all()
    body = out[:heads * plan["tokens"]]
    assert torch.isfinite(body).all()
    for t0, n in zip(plan["row0"], plan["n"]):
        s = body[heads * t0:heads * (t0 + n)].view(heads, n).sum(1)
        assert (s - 1).abs().max().item() < 1e-4

    # the attention alone, all three precisions' routes at head_dim 64
    for prec, parts in ((0, 1), (2, 1), (1, 2)):
        H, D = 6, 384
        e = make_engine(embed_dim=D, heads=H, precision=prec)
        ns = plan["n"]
        M = plan["tokens"]
        g = torch.Generator(device="cuda").manual_seed(11)
        qkv32 = torch.randn(M, 3 * D, generator=g, device="cuda")
        dt = torch.float16 if prec == 2 else torch.bfloat16
        if parts == 2:
            hi = qkv32.to(dt)
            qkv = torch.cat([hi, (qkv32 - hi.float()).to(dt)], 1).contiguous()
            src = qkv32
        else:
            qkv = qkv32.to(dt).contiguous()
            src = qkv.float()
        ctx = torch.full((M + guard, D * parts), float("nan"), device="cuda", dtype=dt)
        tws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
        nt = (C.c_int * len(ns))(*ns)
        check(lib.vitocm_attention_varlen(e, ptr(qkv), qkv.stride(0), len(ns), nt, ptr(ctx), ctx.stride(0), ptr(tws), tws.numel(), cur_stream()))
        torch.cuda.synchronize()
        assert torch.isnan(ctx[M:].float()).all(), prec
        tol = 3e-5 if parts == 2 else 2e-2
        for t0, n in zip(plan["row0"], ns):
            s5 = src[t0:t0 + n].reshape(1, n, 3, H, 64).permute(2, 0, 3, 1, 4)
            ref = attention_reference(s5[0], s5[1], s5[2], 0.125).reshape(n, D)
            got = ctx[t0:t0 + n, :D].float() + (ctx[t0:t0 + n, D:].float() if parts == 2 else 0)
            err = (got - ref).abs().max().item()
            assert err <= tol * max(1.0, ref.abs().max().item()), (prec, n, err)
        lib.vitocm_destroy(e)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_attention_masks_varlen_match_per_image_calls(precision):
    m = _model("tiny", precision)
    sides = [32, 56, 64, 80, 224, 96, 64]
    ims = _images([(s, s) for s in sides], 3, seed=12)
    out = vob.attention_masks_varlen(m, ims, return_attention=True)
    for i, x in enumerate(ims):
        ref = vob.attention_masks(m, x[None], return_attention=True)
        assert torch.equal(out["masks"][i], ref["masks"][0]), i
        assert torch.equal(out["thresholds"][i], ref["thresholds"][0]), i
        assert torch.equal(out["lowres"][i], ref["lowres"][0]), i
        assert torch.equal(out["attention"][i], ref["attention"][0]), i
    # a list of equal-size images equals the tensor call
    same = _images([(64, 64)] * 5, 3, seed=13)
    ref = vob.attention_masks(m, torch.stack(same))
    got = vob.attention_masks_varlen(m, same)
    assert torch.equal(torch.stack(got["masks"]), ref["masks"])
    assert torch.equal(got["thresholds"], ref["thresholds"])
    assert torch.equal(torch.stack(got["lowres"]), ref["lowres"])
    with pytest.raises(ValueError):
        vob.attention_masks_varlen(m, [ims[0], torch.rand(3, 64, 96, device="cuda")])


def test_varlen_refusals():
    m = _model("tiny", "bf16")
    lib = vob._lib.load_library()
    eng = m._ensure_engine()
    x = torch.rand(3 * 64 * 64, device="cuda")
    pos = m._pos_table(64, 64, 64)
    out = torch.empty(2 * 65, device="cuda")
    ws = torch.empty(int(lib.vitocm_varlen_workspace_bytes(eng, 0)), dtype=torch.uint8, device="cuda")
    po = (C.c_int * 1)(0)
    assert lib.vitocm_forward_cls_attn_varlen(eng, ptr(x), 0, 3, (C.c_int * 2)(64, 64), ptr(pos), po, ptr(out), ptr(ws), ws.numel(), 0,
                                              cur_stream()) != 0
    assert lib.vitocm_forward_cls_attn_varlen(eng, ptr(x), 1, 3, (C.c_int * 2)(64, 60), ptr(pos), po, ptr(out), ptr(ws), ws.numel(), 0,
                                              cur_stream()) != 0
    assert b"multiple" in lib.vitocm_last_error()
    assert lib.vitocm_forward_cls_attn_varlen(eng, ptr(x), 1, 3, (C.c_int * 2)(64, 64), ptr(pos), po, ptr(out), ptr(ws), 4096, 0,
                                              cur_stream()) != 0
    assert b"workspace" in lib.vitocm_last_error()
    big = 8 * 256   # 256 x 256 patches: the CLS row (65 537 logits) no longer fits the kernel's shared memory
    assert lib.vitocm_forward_cls_attn_varlen(eng, ptr(x), 1, 3, (C.c_int * 2)(big, big), ptr(pos), po, ptr(out), ptr(ws), ws.numel(), 0,
                                              cur_stream()) != 0
    assert b"shared memory" in lib.vitocm_last_error()
    from functools import partial
    dp = vob.VisionTransformer(img_size=[64], patch_size=8, embed_dim=128, depth=3, num_heads=2, mlp_ratio=4, qkv_bias=True,
                               norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), drop_path_rate=0.1).cuda().train()
    with pytest.raises(vob._lib.VitocmError):
        dp.cls_attention_rows_varlen([x.view(3, 64, 64)])


@pytest.mark.parametrize("n_a", [145, 228, 2181])
def test_varlen_attention_redo_decisions_ignore_the_next_image(n_a):
    """fp16 engine: the first queries of image 1 are built to trip the sum-triggered redo against image 0's keys (their chunk sums of
    exponentials far above 2^14), image 0's own rows are not.  Image 0's ragged last tile holds those queries in its spare rows (no pad
    rows between images); in the call for image 0 alone they are zero rows.  Image 0's CTX must be bit-identical either way.
    145 tokens: the tail is a packed item of the four-pipeline kernel; 228 (a tail of 100 rows) and 2181 (17 full tiles and a tail of 5):
    the tail goes through the two-CTA kernel."""
    H, D, n_b = 6, 384, 200
    e = make_engine(embed_dim=D, heads=H, precision=2)
    lib = vob._lib.load_library()
    g = torch.Generator(device="cuda").manual_seed(21)
    M = n_a + n_b
    qkv = torch.randn(M, 3 * D, generator=g, device="cuda")
    cols = torch.arange(H, device="cuda") * 64          # component 0 of every head
    qkv[:n_a, cols] = 0.0                               # image 0's queries: nothing along it
    qkv[n_a:, cols] = 10.0                              # image 1's queries: large along it ...
    qkv[:128, D + cols] = 0.0                           # ... against image 0's keys beyond the first 128, which are large along it
    qkv[128:n_a, D + cols] = 10.0
    qkv[n_a:, D + cols] = 0.0
    qkv = qkv.half().contiguous()
    ctx = torch.full((M, D), float("nan"), device="cuda", dtype=torch.float16)
    tws = torch.empty(1 << 20, dtype=torch.uint8, device="cuda")
    nt = (C.c_int * 2)(n_a, n_b)
    check(lib.vitocm_attention_varlen(e, ptr(qkv), qkv.stride(0), 2, nt, ptr(ctx), ctx.stride(0), ptr(tws), tws.numel(), cur_stream()))
    for t0, n in ((0, n_a), (n_a, n_b)):
        alone = torch.full((n, D), float("nan"), device="cuda", dtype=torch.float16)
        qi = qkv[t0:t0 + n].contiguous()
        check(lib.vitocm_attention(e, ptr(qi), qi.stride(0), 1, n, ptr(alone), alone.stride(0), cur_stream()))
        torch.cuda.synchronize()
        assert torch.equal(ctx[t0:t0 + n], alone), (n_a, t0, (ctx[t0:t0 + n].float() - alone.float()).abs().max().item())
    lib.vitocm_destroy(e)
