"""GPU (B200): head_dim 128 -- the reference's build_model encoder (embed_dim 384, 3 heads, depth 4) and other models whose heads
are 128 wide.  Kernel level against fp32 torch, model level against the CPU oracle (which takes the head width from its config);
no golden of the reference exists for 3-head models."""
import ctypes as C
from functools import partial

import numpy as np
import pytest
import torch

import vitocm_b200 as vob
from gpu_util import attention_reference, build_model, split_bf16
from oracle import post_oracle as PO
from oracle import train_oracle as TO
from oracle import vit_oracle as VO
from vitocm_b200._lib import VitocmConfig, check, cur_stream, ptr

pytestmark = pytest.mark.gpu

DH = 128
SCALE = DH ** -0.5
REF_CFG = VO.ViTConfig(embed_dim=384, depth=4, num_heads=3, patch_size=8, img_size=224)   # SSS/model.py:91-108


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32 = old


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(*shape, device="cuda", generator=g) * scale


def _engine(heads, precision):
    lib = vob._lib.load_library()
    cfg = VitocmConfig(DH * heads, 1, heads, 4 * DH * heads, 8, 3, 1e-6, SCALE, precision)
    h = C.c_void_p()
    check(lib.vitocm_create(C.byref(cfg), C.byref(h)))
    return h


def _qkv(q, k, v, precision):
    """[B, H, N, 128] x 3 -> the engine's [B*N, 3D] (x 2 parts in fp32-parity mode) activation and the fp32 values it holds"""
    B, H, N, _ = q.shape
    D = DH * H
    qkv32 = torch.stack([q, k, v], 0).permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D).contiguous()
    if precision == 1:
        qkv = split_bf16(qkv32)
        src = qkv[:, :3 * D].float() + qkv[:, 3 * D:].float()
    else:
        qkv = qkv32.to(torch.float16 if precision == 2 else torch.bfloat16).contiguous()
        src = qkv.float()
    return qkv, src.reshape(B, N, 3, H, DH).permute(2, 0, 3, 1, 4)


def _attention(eng, qkv, B, N, D, precision):
    parts = 2 if precision == 1 else 1
    ctx = torch.full((B * N, D * parts), float("nan"), device="cuda", dtype=qkv.dtype)
    check(vob._lib.load_library().vitocm_attention(eng, ptr(qkv), qkv.stride(0), B, N, ptr(ctx), ctx.stride(0), cur_stream()))
    torch.cuda.synchronize()
    return ctx[:, :D].float() + (ctx[:, D:].float() if parts == 2 else 0)


# the shape grid of test_gpu_kernels.test_attention: packed ragged tails of 4 and 2 pairs, none, partly empty last groups
@pytest.mark.parametrize("B,H,N", [(1, 2, 17), (2, 2, 65), (1, 2, 128), (1, 2, 129), (2, 2, 300), (1, 6, 785), (3, 2, 37), (5, 2, 150),
                                   (7, 2, 200), (4, 3, 785), (1, 1, 3137)])
@pytest.mark.parametrize("precision", [0, 1, 2])
def test_attention_head_dim128(B, H, N, precision):
    eng = _engine(H, precision)
    D = DH * H
    q, k, v = (_rand((B, H, N, DH), s) for s in (20, 21, 22))
    qkv, s5 = _qkv(q, k, v, precision)
    ref = attention_reference(s5[0], s5[1], s5[2], SCALE).reshape(B * N, D)
    got = _attention(eng, qkv, B, N, D, precision)
    err = (got - ref).abs().max().item()
    tol = 3e-5 if precision == 1 else 2e-2
    assert err <= tol * max(1.0, ref.abs().max().item()), (err, ref.abs().max().item())
    vob._lib.load_library().vitocm_destroy(eng)


@pytest.mark.parametrize("gain", [6.0, 60.0])
def test_attention_head_dim128_rising_logits_rescale_and_redo(gain):
    """Logits growing along the key axis: lazy rescale of O / l (gain 6) and a redone block (gain 60) on 128-column O."""
    B, H, N = 1, 2, 600
    eng = _engine(H, 0)
    D = DH * H
    q, k, v = (_rand((B, H, N, DH), s) for s in (60, 61, 62))
    k = k * torch.linspace(0.2, 1.0, N, device="cuda").view(1, 1, N, 1) * gain
    qkv, s5 = _qkv(q, k, v, 0)
    ref = attention_reference(s5[0], s5[1], s5[2], SCALE).reshape(B * N, D)
    got = _attention(eng, qkv, B, N, D, 0)
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() <= 3e-2 * max(1.0, ref.abs().max().item())
    vob._lib.load_library().vitocm_destroy(eng)


@pytest.mark.parametrize("B,H,N", [(2, 3, 785), (3, 2, 150), (1, 2, 17), (2, 1, 256)])
def test_attention_backward_head_dim128(B, H, N):
    """LSE rows of the training forward, then dQ / dK / dV against fp32 torch autograd on the bf16-rounded inputs."""
    lib = vob._lib.load_library()
    eng = _engine(H, 0)
    D = DH * H
    qkv = (torch.randn(B * N, 3 * D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(30))).to(torch.bfloat16)
    dctx = (torch.randn(B * N, D, device="cuda", generator=torch.Generator(device="cuda").manual_seed(31)) * 0.5).to(torch.bfloat16)
    src = qkv.float().reshape(B, N, 3, H, DH).permute(2, 0, 3, 1, 4).contiguous().requires_grad_(True)
    logits = (src[0] @ src[1].transpose(-2, -1)) * SCALE
    ctx_ref = (logits.softmax(dim=-1) @ src[2]).transpose(1, 2).reshape(B * N, D)
    ctx_ref.backward(dctx.float())
    dqkv_ref = src.grad.permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D)
    lse_ref = torch.logsumexp(logits, dim=-1).detach() * 1.4426950408889634
    npad = (N + 127) // 128 * 128
    ctx = torch.empty(B * N, D, device="cuda", dtype=torch.bfloat16)
    lse = torch.full((B, H, npad), float("nan"), device="cuda")
    check(lib.vitocm_attention_fwd_lse(eng, ptr(qkv), qkv.stride(0), B, N, ptr(ctx), ctx.stride(0), ptr(lse), cur_stream()))
    torch.cuda.synchronize()
    assert (lse[:, :, :N] - lse_ref).abs().max().item() < 2e-2
    assert torch.isinf(lse[:, :, N:]).all()
    assert (ctx.float() - ctx_ref.detach()).abs().max().item() < 2e-2 * max(1.0, ctx_ref.abs().max().item())
    dqkv = torch.full((B * N, 3 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    delta = torch.empty(B, H, npad, device="cuda")
    dqacc = torch.zeros(B * N, D, device="cuda")
    check(lib.vitocm_attention_bwd(eng, ptr(qkv), qkv.stride(0), ptr(ctx), ptr(dctx), dctx.stride(0), ptr(lse), ptr(delta), ptr(dqacc),
                                   ptr(dqkv), dqkv.stride(0), B, N, cur_stream()))
    torch.cuda.synchronize()
    assert torch.isfinite(dqkv.float()).all()
    assert (dqacc == 0).all(), "dQ accumulator must be left zeroed"
    for name, lo in (("dq", 0), ("dk", D), ("dv", 2 * D)):
        got, ref = dqkv[:, lo:lo + D].float(), dqkv_ref[:, lo:lo + D]
        err = (got - ref).abs().max().item()
        assert err <= 3e-2 * ref.abs().max().item() + 1e-3, (name, err, ref.abs().max().item())
    lib.vitocm_destroy(eng)


def rel_err(a, b):
    return float((np.abs(a - b) / np.abs(b)).max())


@pytest.fixture(scope="module")
def ref_sd():
    return VO.randomize_affine(VO.init_state_dict(REF_CFG, seed=3), seed=4, scale=0.02)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-3), ("bf16", 2e-2), ("fp16", 2e-2)])
def test_reference_encoder_cls_rows(ref_sd, precision, tol):
    m = build_model(REF_CFG, ref_sd, precision, chunk_tiles=2)
    x = VO.synthetic_tile(224, seed=12, batch=3)
    ref = VO.cls_attention_rows(ref_sd, REF_CFG, x).numpy()
    rows = m.cls_attention_rows(x.cuda()).cpu().numpy()
    assert rows.shape == (3, 3, 785)
    assert rel_err(rows, ref) <= tol, rel_err(rows, ref)
    assert np.allclose(rows.sum(-1), 1.0, atol=1e-4)


def test_reference_encoder_query_rows_keys_and_full_attention(ref_sd):
    """attention_rows(..., return_keys=True), get_last_selfattention and get_intermediate_feat at head_dim 128 (fp32-parity)."""
    m = build_model(REF_CFG, ref_sd, "fp32", chunk_tiles=2)
    x = VO.synthetic_tile(224, seed=13, batch=2)
    ref_attn = VO.get_last_selfattention(ref_sd, REF_CFG, x).numpy()
    _, ref_attns, ref_qkvs = VO.get_intermediate_feat(ref_sd, REF_CFG, x, n=1)
    N = ref_attn.shape[-1]
    queries = [0, 1, N // 2, N - 1]
    rows, keys = m.attention_rows(x.cuda(), queries, return_keys=True)
    assert tuple(rows.shape) == (2, 3, 4, N) and tuple(keys.shape) == (2, 3, N, DH)
    assert rel_err(rows.cpu().numpy(), ref_attn[:, :, queries, :]) <= 1e-3
    ref_k = ref_qkvs[0][1].numpy()
    assert np.abs(keys.cpu().numpy() - ref_k).max() <= 1e-4 * max(1.0, np.abs(ref_k).max())
    full = m.get_last_selfattention(x.cuda())
    full = full.materialize() if hasattr(full, "materialize") else full
    assert tuple(full.shape) == (2, 3, N, N)
    assert rel_err(full.cpu().numpy(), ref_attn) <= 1e-3
    _, attns, qkvs = m.get_intermediate_feat(x.cuda(), n=1)
    assert tuple(qkvs[0].shape) == (3, 2, 3, N, DH)
    assert rel_err(attns[0][0, :, N // 2, 1:].cpu().numpy(), ref_attns[0][0, :, N // 2, 1:].numpy()) <= 1e-3


def test_reference_encoder_448_tile(ref_sd):
    """N = 3137: 25 key blocks per query tile, position table resized."""
    m = build_model(REF_CFG, ref_sd, "fp32", chunk_tiles=1)
    x = VO.synthetic_tile(448, seed=44, batch=1)
    ref = VO.cls_attention_rows(ref_sd, REF_CFG, x).numpy()
    rows = m.cls_attention_rows(x.cuda()).cpu().numpy()
    assert rows.shape == (1, 3, 3137)
    assert rel_err(rows, ref) <= 1e-3, rel_err(rows, ref)


def test_reference_encoder_attention_masks(ref_sd):
    """attention_masks in fp32-parity mode against the oracle's post-processing of the oracle's rows.  The masks are integer
    Otsu thresholds of u8 casts of a nearly flat random-init map: where the rows' last digits move the Otsu threshold by one grey
    level, every pixel at that level flips although the rows are within 1e-3 (see test_gpu_parity.py).  So the continuous part is
    held to 99.9 % at the oracle's thresholds, the raw masks to 99.9 % or one threshold step, and the device post-processing of the
    device rows to the oracle's exactly."""
    m = build_model(REF_CFG, ref_sd, "fp32", chunk_tiles=2)
    x = VO.synthetic_tile(224, seed=7, batch=2)
    ref_rows = VO.cls_attention_rows(ref_sd, REF_CFG, x).numpy()
    out = vob.attention_masks(m, x.cuda())
    masks = out["masks"].cpu().numpy()
    rows = m.cls_attention_rows(x.cuda()).cpu().numpy()
    for b in range(2):
        gray = x[b, 0].numpy()
        th, th2, th3, result_ref, att_ref = PO.eval_tile(ref_rows[b], gray, 8)
        g_th, g_th2, g_th3, result, att_u8 = PO.eval_tile(rows[b], gray, 8)
        for i, o in enumerate((g_th, g_th2, g_th3)):
            assert float((masks[b][i] == o).mean()) >= 0.9999
        assert np.abs(result.astype(int) - result_ref.astype(int)).max() <= 1 and np.abs(att_u8.astype(int) - att_ref.astype(int)).max() <= 1
        t_ours, _ = PO.otsu_threshold(result_ref)
        t_heat, _ = PO.otsu_threshold(att_ref)
        fixed = [float(((result > t_ours) == (th > 0)).mean()), float(((att_u8 > t_heat) == (th3 > 0)).mean())]
        assert min(fixed) >= 0.999, fixed
        agree = [float((masks[b][i] == o).mean()) for i, o in enumerate((th, th2, th3))]
        assert agree[1] == 1.0 and min(agree) >= 0.95, agree


def test_reference_encoder_gray_and_mosaic_ingest(ref_sd):
    """CLS rows of single-channel tiles (the gray fast path) and of windows cut out of a uint8 mosaic by the patch embedding,
    MosaicSegmenter on top, and the PGT pseudo-masks, all at head_dim 128."""
    m = build_model(REF_CFG, ref_sd, "fp32", chunk_tiles=3)
    size, W, S = 448, 224, 112
    mosaic = torch.from_numpy(VO.synthetic_mosaic_u8(size, seed=9)).cuda()
    n = vob.grid_size(size, S)
    T = n * n
    x = torch.empty(T, 1, W, W, device="cuda")
    check(vob._lib.load_library().vitocm_extract_tiles(mosaic.data_ptr(), size, size, mosaic.stride(0), n, W, S, 0, T, 1, ptr(x),
                                                       cur_stream()))
    gray = m.cls_attention_rows(x)
    ref = VO.cls_attention_rows(ref_sd, REF_CFG, x.expand(-1, 3, -1, -1).cpu()).numpy()
    assert rel_err(gray.cpu().numpy(), ref) <= 1e-3, rel_err(gray.cpu().numpy(), ref)
    assert torch.equal(m.cls_attention_rows_mosaic(mosaic, n, W, S, 0, T), gray)
    a = vob.MosaicSegmenter(m, window=W, stride=S, tile_batch=3, ingest="direct").segment(mosaic)
    b = vob.MosaicSegmenter(m, window=W, stride=S, tile_batch=3, ingest="crops").segment(mosaic)
    assert torch.equal(a["lowres"], b["lowres"]) and torch.equal(a["th"], b["th"]) and torch.equal(a["th3"], b["th3"])
    y = vob.pgt.pseudo_masks(m, x.expand(-1, 3, -1, -1).contiguous())
    assert tuple(y.shape) == (T, 1, W, W) and set(torch.unique(y).tolist()) <= {0.0, 1.0}


def _key(n):
    return n[len("encoder."):] if n.startswith("encoder.") else n


def _make_mim(cfg_init, img, seed=21):
    sd = VO.randomize_affine(VO.init_state_dict(cfg_init, seed=seed, mim=True), seed=seed + 1)
    gd = torch.Generator().manual_seed(seed + 2)
    D = cfg_init.embed_dim
    dec_w, dec_b = torch.randn(192, D, 1, 1, generator=gd) * 0.05, torch.randn(192, generator=gd) * 0.05
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=D, depth=cfg_init.depth, num_heads=cfg_init.num_heads, mlp_ratio=4,
                                         img_size=[img], qkv_bias=True, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision="bf16")
    enc.load_state_dict(sd, strict=True)
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    mim.decoder[0].weight.data.copy_(dec_w)
    mim.decoder[0].bias.data.copy_(dec_b)
    params = dict(sd)
    params["decoder.0.weight"], params["decoder.0.bias"] = dec_w, dec_b
    return mim.cuda().train(), params


def test_mim_two_steps_track_train_oracle():
    """Two MIM steps (loss.sum().backward(), clip_grad_norm_, AdamW) of a 2-head x 128 model against train_oracle, with the bars
    of test_gpu_train.py."""
    cfg_init = VO.ViTConfig(embed_dim=256, depth=2, num_heads=2, patch_size=8, img_size=224)
    cfg = VO.ViTConfig(embed_dim=256, depth=2, num_heads=2, patch_size=8, img_size=32)
    mim, params = _make_mim(cfg_init, 32)
    groups = vob.optimizer.get_pretrain_param_groups(mim, None, mim.no_weight_decay(), mim.no_weight_decay_keywords())
    opt = torch.optim.AdamW(groups, eps=1e-8, betas=(0.9, 0.999), lr=5e-4, weight_decay=0.05)
    state = TO.TrainState({k: v.clone() for k, v in params.items()})
    rs = np.random.RandomState(8)
    for it, clip in ((0, 5.0), (1, 0.05)):
        x = VO.synthetic_tile(32, seed=50 + it, batch=4)
        mask = torch.from_numpy(np.stack([VO.mask_generator(rs, 32, 16, 8, 0.5) for _ in range(4)]))
        ref_loss, ref_norm, ref = TO.train_step(state, cfg, x, mask, clip_grad=clip)   # ref: the clipped gradients
        opt.zero_grad()
        loss, _, _ = mim(x.cuda(), mask.cuda())
        loss.sum().backward()
        assert abs(loss.item() - ref_loss.item()) <= 2e-2 * abs(ref_loss.item())
        total = torch.nn.utils.clip_grad_norm_(mim.parameters(), clip)
        assert abs(total.item() - ref_norm.item()) <= 2e-2 * ref_norm.item()
        num = den = 0.0
        for n, p in mim.named_parameters():
            r = ref[_key(n)]
            num += float((p.grad.cpu() - r).double().pow(2).sum())
            den += float(r.double().pow(2).sum())
        # step 1 starts from parameters that already differ (Adam's first update is ~lr * sign(g)): looser bar, as in test_gpu_train.py
        assert (num / den) ** 0.5 <= (3e-2 if it == 0 else 1.5e-1), (num / den) ** 0.5
        opt.step()
        for n, p in mim.named_parameters():
            assert (p.detach().cpu() - state.params[_key(n)]).abs().max().item() <= 2.5 * 5e-4 * (it + 1), n


def test_reference_encoder_mim_batch32_loss_decreases():
    """build_model(args, depth=4, num_heads=3) -- the reference's encoder -- one batch of 32 224^2 tiles, a few fused AdamW steps."""
    from types import SimpleNamespace as NS
    args = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=224),
              TRAIN=NS(BASE_LR=5e-4, WEIGHT_DECAY=0.05, OPTIMIZER=NS(NAME="adamw", EPS=1e-8, BETAS=(0.9, 0.999))))
    torch.manual_seed(0)
    enc = vob.model.build_model(args, depth=4, num_heads=3)
    assert enc.embed_dim // enc.num_heads == 128 and enc.depth == 4
    mim = vob.MIM(encoder=enc, encoder_stride=8).cuda().train()
    opt = vob.optimizer.build_pretrain_optimizer(args, mim, None)
    x = VO.synthetic_tile(224, seed=77, batch=32).cuda()
    rs = np.random.RandomState(3)
    mask = torch.from_numpy(np.stack([VO.mask_generator(rs, 224, 32, 8, 0.6) for _ in range(32)])).cuda()
    losses = []
    for _ in range(4):
        opt.zero_grad()
        loss, _, _ = mim(x, mask)
        loss.sum().backward()
        vob.optimizer.clip_grad_norm_(mim.parameters(), 5.0)
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)), losses
    assert losses[-1] < losses[0], losses
