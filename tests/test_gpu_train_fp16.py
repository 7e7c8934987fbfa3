"""GPU (B200): MIM training on fp16 engines -- the fp16 weight-gradient GEMM and attention backward through the C ABI, the whole
step against the float64 oracle next to the same step on a bf16 engine, and the power-of-two loss scale of the fp16 backward."""
from functools import partial
from types import SimpleNamespace as NS

import numpy as np
import pytest
import torch

import vitocm_b200 as vob
from gpu_util import make_engine
from oracle import train_oracle as TO
from oracle import vit_oracle as VO
from vitocm_b200._lib import check, cur_stream, ptr

pytestmark = pytest.mark.gpu

FP16 = 2


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield


def _rand(shape, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda") * scale


def _key(n):
    return n[len("encoder."):] if n.startswith("encoder.") else n


# ---------------------------------------------------------------------------------------------------------- kernel level
@pytest.mark.parametrize("M,R,C", [(50, 72, 64), (333, 64, 256), (785, 192, 384), (1570, 1152, 384), (3000, 384, 768),
                                   (1568, 384, 192), (20000, 128, 128), (100, 128, 576)])
def test_wgrad_fp16(M, R, C):
    """dW += G^T A and the bias column (all-ones MMA, fp16 1.0) on an fp16 engine, against float64 on the same fp16 values."""
    lib = vob._lib.load_library()
    eng = make_engine(precision=FP16)
    G = _rand((M, R), 1, 0.5).half()
    A = _rand((M, C), 2).half()
    dW0, db0 = _rand((R, C), 3), _rand((R,), 6)
    dW, db = dW0.clone(), db0.clone()
    check(lib.vitocm_wgrad(eng, ptr(G), G.stride(0), ptr(A), A.stride(0), M, R, C, ptr(dW), ptr(db), cur_stream()))
    torch.cuda.synchronize()
    ref = dW0.double() + G.double().T @ A.double()
    assert (dW.double() - ref).abs().max().item() <= 2e-5 * ref.abs().max().item() + 1e-4
    ref_b = db0.double() + G.double().sum(0)
    assert (db.double() - ref_b).abs().max().item() <= 2e-5 * ref_b.abs().max().item() + 1e-4
    lib.vitocm_destroy(eng)


def _attention_f64(qkv, dctx, B, H, N, dh, scale):
    """float64 autograd of vit.py:83-87 on the fp32 inputs -> dqkv [B*N][3D]"""
    D = dh * H
    src = qkv.double().reshape(B, N, 3, H, dh).permute(2, 0, 3, 1, 4).contiguous().requires_grad_(True)
    q, k, v = src[0], src[1], src[2]
    a = ((q @ k.transpose(-2, -1)) * scale).softmax(dim=-1)
    ctx = (a @ v).transpose(1, 2).reshape(B * N, D)
    ctx.backward(dctx.double())
    return src.grad.permute(1, 3, 0, 2, 4).reshape(B * N, 3 * D)


def _attention_bwd_errors(precision, qkv32, dctx32, B, H, N, dh, ref):
    lib = vob._lib.load_library()
    D = dh * H
    eng = make_engine(embed_dim=D, heads=H, precision=precision)
    dt = torch.float16 if precision == FP16 else torch.bfloat16
    qkv, dctx = qkv32.to(dt), dctx32.to(dt)
    npad = (N + 127) // 128 * 128
    ctx = torch.empty(B * N, D, device="cuda", dtype=dt)
    lse = torch.empty(B, H, npad, device="cuda")
    check(lib.vitocm_attention_fwd_lse(eng, ptr(qkv), qkv.stride(0), B, N, ptr(ctx), ctx.stride(0), ptr(lse), cur_stream()))
    dqkv = torch.full((B * N, 3 * D), float("nan"), device="cuda", dtype=dt)
    delta = torch.empty(B, H, npad, device="cuda")
    dqacc = torch.zeros(B * N, D, device="cuda")
    check(lib.vitocm_attention_bwd(eng, ptr(qkv), qkv.stride(0), ptr(ctx), ptr(dctx), dctx.stride(0), ptr(lse), ptr(delta), ptr(dqacc),
                                   ptr(dqkv), dqkv.stride(0), B, N, cur_stream()))
    torch.cuda.synchronize()
    lib.vitocm_destroy(eng)
    assert (dqacc == 0).all(), "dQ accumulator must be left zeroed"
    assert torch.isfinite(dqkv.float()).all()
    errs = {}
    for name, lo in (("dq", 0), ("dk", D), ("dv", 2 * D)):
        r = ref[:, lo:lo + D]
        errs[name] = (dqkv[:, lo:lo + D].double() - r).abs().max().item() / r.abs().max().item()
    return errs


@pytest.mark.parametrize("B,H,N,dh", [(2, 6, 17, 64), (3, 6, 145, 64), (2, 6, 785, 64), (32, 6, 785, 64),
                                      (2, 3, 785, 128), (32, 3, 785, 128)])
def test_attention_backward_fp16_beats_bf16(B, H, N, dh):
    """The fp16 attention backward (both head widths, ragged tails, persistent CTAs walking many items) against float64 autograd of
    the unrounded inputs; the same inputs through a bf16 engine must come out further from it."""
    D = dh * H
    qkv = _rand((B * N, 3 * D), 30)
    dctx = _rand((B * N, D), 31, 0.5)
    scale = 0.125      # make_engine's qk scale
    ref = _attention_f64(qkv, dctx, B, H, N, dh, scale)
    e16 = _attention_bwd_errors(FP16, qkv, dctx, B, H, N, dh, ref)
    ebf = _attention_bwd_errors(0, qkv, dctx, B, H, N, dh, ref)
    print(f"B={B} H={H} N={N} head_dim={dh}: max error / max |ref|  fp16 {e16}  bf16 {ebf}")
    for name in e16:
        assert e16[name] < ebf[name], (name, e16[name], ebf[name])
        assert e16[name] <= 6e-3, (name, e16[name])


# ---------------------------------------------------------------------------------------------------------- MIM step
def _make_mim(cfg_init, img, precision, seed):
    sd = VO.randomize_affine(VO.init_state_dict(cfg_init, seed=seed, mim=True), seed=seed + 1)
    gd = torch.Generator().manual_seed(seed + 2)
    D = cfg_init.embed_dim
    dec_w, dec_b = torch.randn(192, D, 1, 1, generator=gd) * 0.05, torch.randn(192, generator=gd) * 0.05
    enc = vob.VisionTransformerForSimMIM(patch_size=8, embed_dim=D, depth=cfg_init.depth, num_heads=cfg_init.num_heads, mlp_ratio=4,
                                         img_size=[img], qkv_bias=True, norm_layer=partial(torch.nn.LayerNorm, eps=1e-6), precision=precision)
    enc.load_state_dict(sd, strict=True)
    mim = vob.MIM(encoder=enc, encoder_stride=8)
    mim.decoder[0].weight.data.copy_(dec_w)
    mim.decoder[0].bias.data.copy_(dec_b)
    params = dict(sd)
    params["decoder.0.weight"], params["decoder.0.bias"] = dec_w, dec_b
    return mim.cuda().train(), params


def _grad_errors(mim, ref):
    num = den = 0.0
    worst = ("", 0.0)
    for n, p in mim.named_parameters():
        r = ref[_key(n)].double().cuda()
        d = p.grad.double() - r
        num += d.pow(2).sum().item()
        den += r.pow(2).sum().item()
        err = d.abs().max().item() / max(r.abs().max().item(), 1e-8)
        if err > worst[1]:
            worst = (n, err)
    return (num / den) ** 0.5, worst


def _step_vs_oracle(cfg_init, cfg, img, batch, seed, scale_linear=1.0):
    x = VO.synthetic_tile(img, seed=seed + 5, batch=batch)
    rs = np.random.RandomState(seed + 6)
    mask = torch.from_numpy(np.stack([VO.mask_generator(rs, img, 32 if img % 32 == 0 else 8, 8, 0.6) for _ in range(batch)]))
    out = {}
    ref_loss = ref = None
    for precision in ("bf16", "fp16"):
        mim, params = _make_mim(cfg_init, img, precision, seed)
        if scale_linear != 1.0:   # every Linear weight (and the decoder's 1 x 1 conv) x scale_linear
            with torch.no_grad():
                for n, p in mim.named_parameters():
                    if n.endswith(".weight") and p.dim() >= 2 and "patch_embed" not in n:
                        p.mul_(scale_linear)
                        params[_key(n)] = params[_key(n)] * scale_linear
        if ref is None:
            ref_loss, ref = TO.mim_loss_and_grads({k: v.double().cuda() for k, v in params.items()}, cfg, x.double().cuda(), mask.cuda())
        loss, _, _ = mim(x.cuda(), mask.cuda())
        loss.sum().backward()
        for n, p in mim.named_parameters():
            assert torch.isfinite(p.grad).all(), (precision, n)
        out[precision] = (loss.item(), *_grad_errors(mim, ref))
        del mim
    return ref_loss.item(), out


# (ViT-S/8 at batch 2, 32 and 84, the reference's encoder, ViT-B width at 64^2, N = 5): fp16 against bf16 on the same inputs.  At
# batch 84 M = 65 940 tokens, so fc1 and the input gradient through the GELU run on CTA pairs (BN 192 at D = 384, 256 at D = 128).
@pytest.mark.parametrize("D,heads,depth,img,batch", [pytest.param(384, 6, 12, 224, 2, id="vit-small-b2"),
                                                     pytest.param(384, 6, 2, 224, 32, id="vit-small-b32"),
                                                     pytest.param(384, 6, 2, 224, 84, id="vit-small-b84"),
                                                     pytest.param(128, 2, 2, 224, 84, id="d128-b84"),
                                                     pytest.param(384, 3, 4, 224, 32, id="reference-encoder-b32"),
                                                     pytest.param(768, 12, 2, 64, 3, id="vit-base-width-64px"),
                                                     pytest.param(128, 2, 2, 16, 4, id="n5")])
def test_fp16_step_closer_to_oracle_than_bf16(D, heads, depth, img, batch):
    cfg_init = VO.ViTConfig(embed_dim=D, depth=depth, num_heads=heads, patch_size=8, img_size=224)
    cfg = VO.ViTConfig(embed_dim=D, depth=depth, num_heads=heads, patch_size=8, img_size=img)
    ref_loss, out = _step_vs_oracle(cfg_init, cfg, img, batch, seed=70 + heads + depth)
    (l16, g16, w16), (lbf, gbf, wbf) = out["fp16"], out["bf16"]
    print(f"D={D} heads={heads} depth={depth} img={img} batch={batch}: loss oracle {ref_loss:.6f} fp16 {l16:.6f} bf16 {lbf:.6f}; "
          f"global relative L2 gradient error fp16 {g16:.3e} bf16 {gbf:.3e}; worst tensor fp16 {w16[1]:.3e} ({w16[0]}) "
          f"bf16 {wbf[1]:.3e} ({wbf[0]})")
    assert abs(l16 - ref_loss) <= 2e-3 * abs(ref_loss)
    assert g16 < gbf
    assert g16 <= (1e-2 if batch * (img // 8) ** 2 >= 64 else 3e-2)


def test_fp16_step_with_linear_weights_times_4():
    """Range stress: every Linear weight x4 grows the activations and the backward's intermediate gradients; the loss scale must
    leave room for them (finite gradients, still on the oracle)."""
    cfg = VO.ViTConfig(embed_dim=384, depth=4, num_heads=3, patch_size=8, img_size=224)
    ref_loss, out = _step_vs_oracle(cfg, cfg, 224, 32, seed=90, scale_linear=4.0)
    (l16, g16, w16), (lbf, gbf, _) = out["fp16"], out["bf16"]
    print(f"weights x4: loss oracle {ref_loss:.6f} fp16 {l16:.6f} bf16 {lbf:.6f}; global relative L2 gradient error fp16 {g16:.3e} "
          f"bf16 {gbf:.3e}; worst tensor fp16 {w16[1]:.3e} ({w16[0]})")
    assert g16 <= 2e-2


def _grads_at(mim, x, mask, gscale):
    mim.zero_grad(set_to_none=True)
    loss, _, _ = mim(x, mask)
    (loss * gscale).sum().backward()
    return mim._gflat.clone()


def test_loss_scale_is_exact_for_power_of_two_grad_scale():
    """The backward of gscale * loss for gscale = 2^-24 ... 2^16 gives gscale x the gscale = 1 gradients: the loss scale absorbs the power
    of two, so every 16-bit tensor of the backward holds the same bits (without a loss scale 2^-24 would flush every gradient to 0).
    The fp32 reductions that combine partial sums with atomics may order them differently from run to run; the bar is that run-to-run
    spread, measured by repeating the gscale = 1 backward."""
    cfg_init = VO.ViTConfig(embed_dim=384, depth=2, num_heads=3, patch_size=8, img_size=224)
    mim, _ = _make_mim(cfg_init, 64, "fp16", seed=50)
    x = VO.synthetic_tile(64, seed=51, batch=4).cuda()
    rs = np.random.RandomState(52)
    mask = torch.from_numpy(np.stack([VO.mask_generator(rs, 64, 16, 8, 0.5) for _ in range(4)])).cuda()
    g1 = _grads_at(mim, x, mask, 1.0)
    spread = (_grads_at(mim, x, mask, 1.0) - g1).abs().max().item()
    assert g1.abs().max().item() > 0
    for e in (-24, -8, 8, 16):
        g = _grads_at(mim, x, mask, 2.0 ** e)
        assert torch.isfinite(g).all()
        diff = (g * 2.0 ** -e - g1).abs().max().item()
        print(f"gscale 2^{e}: max |grad / gscale - grad(1)| = {diff:.3e} (run-to-run spread {spread:.3e}); bitwise {diff == 0.0}")
        assert diff <= 2 * spread + 1e-7 * g1.abs().max().item(), (e, diff, spread)


def test_fp16_gradient_accumulation():
    """Two backwards without zero_grad accumulate into the sum of the single ones (mim.py:160-171)."""
    cfg_init = VO.ViTConfig(embed_dim=128, depth=2, num_heads=2, patch_size=8, img_size=224)
    mim, _ = _make_mim(cfg_init, 32, "fp16", seed=21)
    xs = [VO.synthetic_tile(32, seed=40 + k, batch=2).cuda() for k in range(2)]
    rs = np.random.RandomState(7)
    ms = [torch.from_numpy(np.stack([VO.mask_generator(rs, 32, 16, 8, 0.5) for _ in range(2)])).cuda() for _ in range(2)]
    singles = [_grads_at(mim, x, m, 0.5) for x, m in zip(xs, ms)]
    mim.zero_grad(set_to_none=True)
    for x, m in zip(xs, ms):
        loss, _, _ = mim(x, m)
        (loss / 2).sum().backward()
    want = singles[0] + singles[1]
    assert (mim._gflat - want).abs().max().item() <= 1e-5 * want.abs().max().item() + 1e-7


def test_fp16_reference_encoder_trains_and_cls_rows_track_oracle():
    """build_model(args, depth=4, num_heads=3, precision="fp16") through the reference loop with FusedAdamW and clip: the loss falls
    over five steps on one batch of 32, and the CLS rows of the same fp16 engine after the steps match the oracle's for the updated
    weights."""
    args = NS(MODEL=NS(PATCH_SIZE=8), DATA=NS(IMG_SIZE=224),
              TRAIN=NS(BASE_LR=5e-4, WEIGHT_DECAY=0.05, OPTIMIZER=NS(NAME="adamw", EPS=1e-8, BETAS=(0.9, 0.999))))
    torch.manual_seed(0)
    enc = vob.model.build_model(args, depth=4, num_heads=3, precision="fp16")
    mim = vob.MIM(encoder=enc, encoder_stride=8).cuda().train()
    opt = vob.optimizer.build_pretrain_optimizer(args, mim, None)
    x = VO.synthetic_tile(224, seed=77, batch=32).cuda()
    rs = np.random.RandomState(3)
    mask = torch.from_numpy(np.stack([VO.mask_generator(rs, 224, 32, 8, 0.6) for _ in range(32)])).cuda()
    losses = []
    for _ in range(5):
        opt.zero_grad()
        loss, _, _ = mim(x, mask)
        loss.sum().backward()
        vob.optimizer.clip_grad_norm_(mim.parameters(), 5.0)
        opt.step()
        losses.append(loss.item())
    print("fp16 reference encoder, losses:", losses)
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    mim.eval()
    xe = VO.synthetic_tile(224, seed=78, batch=3)
    sd = {k: v.detach().cpu() for k, v in mim.encoder.state_dict().items()}
    cfg = VO.ViTConfig(embed_dim=384, depth=4, num_heads=3, patch_size=8, img_size=224)
    ref = VO.cls_attention_rows(sd, cfg, xe).numpy()
    rows = mim.encoder.cls_attention_rows(xe.cuda()).cpu().numpy()
    err = float((np.abs(rows - ref) / ref).max())
    print(f"CLS rows after 5 fp16 steps: max relative error {err:.3e}")
    assert err <= 2e-2
